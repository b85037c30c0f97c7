#!/usr/bin/env python3
"""Benchmark of the Polya-Gamma hot path (bench contract: see the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl engine|reference]
                    [--workload hybrid|pg1] [--num DRAWS | --draws DRAWS] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], SURVEY.md section 8d "C2"): 100M mixed-shape
PG(b,z) draws per GPU -- b: 50% real U(0.5,200), 50% integer U{1..200};
z ~ U(-5,5); seed 20240002 -- exercising the Devroye / sum-of-gammas / alternate /
saddle-point / normal dispatch of rpg_hybrid (LogitWrapper.cpp:129-167).
A step is one pass of rpg_hybrid over the whole batch.

  value  : draws/s with inputs resident in HBM (CUDA events on the launch stream)
  e2e    : draws/s through the reference-facing C ABI `rpg_hybrid` with pinned HOST
           buffers, H2D + D2H inside the timed region
  roofline, cpu_baseline, clocks, gpu_launches: see DESIGN.md "Measurement"

`--impl reference` times the reference's own CPU sampler (oracle/_ref: the
reference sources compiled in place; the plain-C port if that is absent) on all
host cores, on a bounded sample of the same workload.

N > 1: one process per GPU under torchrun; observations are sharded, rank r draws
global observations [r*num, (r+1)*num) -- no data-path collective ("weak").

--dump-outputs DIR writes the draws of the last timed step to DIR/omega.npy (float64;
DIR/omega_rank<r>.npy per rank under torchrun), so that two builds can be compared draw
for draw on the same inputs.  A batch larger than DUMP_DRAWS is sampled: one draw from
each of DUMP_DRAWS equal strata, at offsets drawn from a fixed seed.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20240002
CPU_SAMPLE = {"hybrid": 16_000_000, "pg1": 64_000_000}
# algorithmic HBM bytes per draw: shape in + z in + omega out (fp64; n is int32 for pg1)
BYTES_PER_DRAW = {"hybrid": 24, "pg1": 20}
# fp64-equivalent flop model per draw, SURVEY.md section 8(d): 0.9 kFLOP for a Devroye
# PG(1,z) draw; the mixed workload is weighted by its regime shares (SP ~ 10x).
KFLOP_PER_DRAW = {"pg1": 0.9, "hybrid": 0.786 * 9.0 + 0.058 * 3.0 + 0.15 * 0.3 + 0.005 * 1.35 + 0.0013 * 60.0}
DUMP_DRAWS = 4 << 20            # 32 MB of fp64 draws per run, over all ranks


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="hybrid", choices=["hybrid", "pg1"])
    # --draws: the same under torchrun, whose own parser rejects "--num" as an ambiguous prefix of --numa-binding
    ap.add_argument("--num", "--draws", dest="num", type=int, default=100_000_000, help="draws per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the PG(1,z) and logit-Gibbs extras")
    ap.add_argument("--gibbs-iters", type=int, default=200)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the draws of the last timed step to DIR/omega.npy")
    return ap.parse_args()


def dump_index(num, world=1):
    """Which of a rank's num draws --dump-outputs writes: None for all of them, else the fixed
    stratified sample the module docstring describes."""
    import numpy as np
    k = DUMP_DRAWS // world
    if num <= k:
        return None
    rng = np.random.default_rng([SEED, num])
    return np.arange(k, dtype=np.int64) * num // k + rng.integers(0, num // k, k)


def dump_outputs(directory, name, x):
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, name + ".npy"), np.asarray(x, dtype=np.float64))


def make_inputs_numpy(workload, num, obs0=0):
    """The workload's (shape, z) for global observations [obs0, obs0+num) -- host side."""
    import numpy as np
    rng = np.random.default_rng([SEED, obs0])
    z = rng.uniform(-5.0, 5.0, num)
    if workload == "pg1":
        return np.ones(num, dtype=np.int32), z
    real = rng.uniform(0.5, 200.0, num)
    integer = rng.integers(1, 201, num).astype(np.float64)
    return np.where(rng.random(num) < 0.5, real, integer), z


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.QUERY,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [t.strip() for t in line.split(",")]))

    def stop(self, t0, t1, tw=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        # a row is stamped when it is READ, up to one polling period after nvidia-smi sampled it
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.1]
        window = "timed steps"
        if len(rows) < 2 and tw is not None:     # a timed region shorter than two polling periods
            rows = [r for t, r in self.rows if tw <= t <= t1 + 0.1]
            window = "warm-up + timed steps (same kernels, back to back)"
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        def num(v):                                   # nvidia-smi prints "[N/A]" for fields a board lacks
            try:
                return float(v)
            except (TypeError, ValueError):
                return None
        sm = sorted(v for v in (num(r[1]) for r in rows if len(r) > 2) if v is not None)
        pw = [v for v in (num(r[3]) for r in rows if len(r) > 3) if v is not None]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 5 + k and r[5 + k] == "Active" for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": num(rows[0][2]) if len(rows[0]) > 2 else None,
                "reasons": reasons, "samples": len(rows), "window": window, "power_w_max": max(pw) if pw else None}


def load_oracle():
    from oracle import loader
    if loader.available("reference"):
        return loader.Oracle("reference")
    if not loader.available("port"):
        loader.build(("port",))
    return loader.Oracle("port")


def time_cpu(workload, sample, nthreads):
    """Reference CPU sampler on `sample` draws of the workload; returns (seconds, kind, draws)."""
    O = load_oracle()
    shape, z = make_inputs_numpy(workload, sample)
    t = time.perf_counter()
    if workload == "pg1":
        x = O.rpg_devroye(shape, z, seed=SEED, nthreads=nthreads)
    else:
        x = O.rpg_hybrid(shape, z, seed=SEED, nthreads=nthreads)
    return time.perf_counter() - t, O.kind, x


def measured_pipe_peaks(L):
    """Pipe throughputs of THIS device, measured now (bl_probe_peaks): the denominators of the compute roofline."""
    import ctypes as C
    from bayeslogit_b200 import _lib
    b = (C.c_double * 6)()
    _lib.check(L.bl_probe_peaks(C.cast(b, C.c_void_p)))
    v = list(b)
    return {"fp64_fma_tflops": v[0], "fp32_fma_tflops": v[1], "mufu_gops": v[2], "fp64_tensor_dmma_tflops": v[3],
            "imad_wide_gops": v[4],
            # warp instructions issued per second: the better of the mixed FFMA + IMAD kernel and the FFMA kernel
            # (one FFMA warp instruction = 64 flop)
            "issue_gwarp_inst": max(v[5], v[1] * 1e3 / 64.0),
            "how": "bl_probe_peaks (bayeslogit_b200/csrc/probe_peaks.cu): 8 independent chains per thread, 2 x 1024 threads "
                   "per SM, best of 4 launches, in this run at this run's clocks"}


def cpu_gibbs_baseline(N, P, iters_all, iters_one):
    """Logit::gibbs_block (Logit.hpp:402-457) restated on the host cores (oracle/gibbs_oracle.c: psi, draw_w through the
    port sampler, the sqrt(w)-scaled Gram, both beta draws), timed on the C3 shape: all host threads (OpenMP) and one."""
    import numpy as np
    from oracle import loader
    rng = np.random.default_rng(20240003)
    X = np.c_[rng.standard_normal((N, P - 1)), np.ones(N)]
    bt = np.r_[np.abs(rng.normal(0, 0.25, P - 1)), -0.5]
    y = (rng.random(N) < 1.0 / (1.0 + np.exp(-X @ bt))).astype(np.float64)
    n = np.ones(N)
    m0, P0 = np.zeros(P), 0.01 * np.eye(P)
    cores = os.cpu_count() or 1
    out = {"N": N, "P": P, "cores": cores, "kind": "port",
           "what": "oracle/gibbs_oracle.c pgb_logit_gibbs = restatement of Logit::gibbs_block (the reference's model layer "
                   "needs the absent Matrix/BLAS libraries); plain loops, OpenMP over observations"}
    for label, constrained in (("plain_beta", False), ("reference_constrained_beta", True)):
        loader.logit_gibbs(y, X, n, m0, P0, 1, 1, seed=1, constrained=constrained, nthreads=cores)      # warm-up
        t = time.perf_counter()
        loader.logit_gibbs(y, X, n, m0, P0, 1, iters_all - 1, seed=20240003, constrained=constrained, nthreads=cores)
        dt_all = time.perf_counter() - t
        t = time.perf_counter()
        loader.logit_gibbs(y, X, n, m0, P0, 1, iters_one - 1, seed=20240003, constrained=constrained, nthreads=1)
        dt_one = time.perf_counter() - t
        out[label] = {"iters_per_sec_all_cores": iters_all / dt_all, "iters_all_cores": iters_all,
                      "iters_per_sec_1_core": iters_one / dt_one, "iters_1_core": iters_one}
    return out


def bind_to_gpu_numa_node(local):
    """Multi-rank runs: keep this rank's host threads -- and with them the first-touch placement of its pinned
    buffers and the library's copy threads -- on the NUMA node its GPU hangs off, so that the ranks' host-side
    traffic does not cross sockets.  Returns the node, or None when the topology cannot be read."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except (OSError, ValueError, AttributeError):
        return None


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sample = min(CPU_SAMPLE[args.workload], args.num)
    for _ in range(args.warmup):
        time_cpu(args.workload, max(sample // 16, 1), cores)
    t = 0.0
    kind = "port"
    for _ in range(args.steps):
        dt, kind, x = time_cpu(args.workload, sample, cores)
        t += dt
    if args.dump_outputs:
        idx = dump_index(sample)
        dump_outputs(args.dump_outputs, "omega", x if idx is None else x[idx])
    value = sample * args.steps / t
    desc = f"first {sample} draws of the workload per step, all {cores} host threads (OpenMP, one RNG+sampler per thread)"
    one = max(sample // 8, 1)
    dt1, _, _ = time_cpu(args.workload, one, 1)
    print(json.dumps({
        "impl": "reference", "metric": "pg_draws_per_sec", "value": value, "unit": "draws/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": dict(workload_config(args), timed_sample_per_step=sample,
                       note="a rate: each step draws the first timed_sample_per_step observations of the workload"),
        "cpu_baseline": {"value": value, "unit": "draws/s", "cores": cores, "kind": kind, "sample": desc,
                         "value_1_core": one / dt1,
                         "sample_1_core": f"first {one} draws, one thread (the reference's shipped serial loop, "
                                          f"LogitWrapper.cpp:129-167)"},
        "e2e": {"value": value, "unit": "draws/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(args):
    name = ("rpg_hybrid mixed-shape PG(b,z): b 50% real U(0.5,200) + 50% integer U{1..200}, z~U(-5,5)"
            if args.workload == "hybrid" else "rpg_devroye PG(1,z), z~U(-5,5)")
    return {"workload": name, "draws_per_gpu_per_step": args.num, "seed": SEED,
            "l2": "inputs_larger_than_l2" if args.num * 16 > 126e6 else "l2_flushed_between_steps",
            "parallelism": f"obs-shard x{args.gpus}"}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    # Exactly ONE line on stdout: native libraries write there too (NCCL prints its version banner on
    # rank 0 when NCCL_DEBUG is set), so file descriptor 1 points at stderr for the duration of the run
    # and the JSON line goes to the saved descriptor at the end.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import numpy as np
    import torch
    import torch.distributed as dist
    from bayeslogit_b200 import _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_node = bind_to_gpu_numa_node(local) if world > 1 else None
    L = _lib.lib()
    _lib.check(L.bl_set_device(local))
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    pipe_peaks = measured_pipe_peaks(L)
    num = args.num
    obs0 = rank * num
    wl = args.workload
    shape_h, z_h = make_inputs_numpy(wl, num, obs0)
    # device-resident inputs for `value`
    shape_d = torch.from_numpy(shape_h).to(dev)
    z_d = torch.from_numpy(z_h).to(dev)
    x_d = torch.empty(num, dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if num * 16 <= 126e6 else None
    stream = torch.cuda.current_stream().cuda_stream
    fn_dev = L.bl_rpg_hybrid_dev if wl == "hybrid" else L.bl_rpg_devroye_dev

    def step_dev(call):
        if flush is not None:
            flush.zero_()
        st = fn_dev(x_d.data_ptr(), shape_d.data_ptr(), z_d.data_ptr(), num, SEED, call, obs0, stream)
        if st:
            _lib.check(st)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing ----------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        time.sleep(0.5)                                  # nvidia-smi start-up: first row after ~0.3 s
    t_warm0 = time.time()
    for w in range(args.warmup):
        step_dev(1000 + w)
    barrier()
    launches0 = L.bl_kernel_launches()
    t_wall0 = time.time()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    kern_ms = 0.0
    ev[0].record()
    for k in range(args.steps):
        if flush is not None:
            flush.zero_()
            e_a = torch.cuda.Event(enable_timing=True); e_a.record()
        st = fn_dev(x_d.data_ptr(), shape_d.data_ptr(), z_d.data_ptr(), num, SEED, k, obs0, stream)
        if st:
            _lib.check(st)
        ev[k + 1].record()
        if flush is not None:
            ev[k + 1].synchronize()
            kern_ms += e_a.elapsed_time(ev[k + 1])
    barrier()
    t_wall1 = time.time()
    launches = L.bl_kernel_launches() - launches0
    total_ms = max_over_ranks(ev[0].elapsed_time(ev[-1]))
    if flush is None:
        kern_ms = ev[0].elapsed_time(ev[-1])
    kern_ms = max_over_ranks(kern_ms) / args.steps       # dominant kernel, per launch
    clocks = sampler.stop(t_wall0, t_wall1, t_warm0) if sampler else None
    value = world * num * args.steps / (total_ms * 1e-3)
    mean_omega = float(x_d[: 1 << 20].mean().item())
    if args.dump_outputs:            # now: the passes below overwrite x_d
        idx = dump_index(num, world)
        x = x_d if idx is None else x_d[torch.from_numpy(idx).to(dev)]
        dump_outputs(args.dump_outputs, "omega" if world == 1 else f"omega_rank{rank}", x.cpu().numpy())
    # dominant kernel of the step, timed live with CUDA events on the launch stream (separate,
    # untimed pass so the event records do not sit inside the headline region)
    stage_ms, stage_launches, regime_counts = None, None, None
    if wl == "hybrid":
        import ctypes as C
        names = ["binning", "sp_setup", "sp_loop", "alt_setup", "alt_loop", "sum_of_gammas", "normal", "devroye"]
        L.bl_hybrid_timing(1)
        acc = [0.0] * 8
        nl = [0] * 8
        reps = max(1, min(3, args.steps))
        for k in range(reps):
            step_dev(3000 + k)
            buf, cnt = (C.c_double * 8)(), (C.c_int * 8)()
            if L.bl_hybrid_timing_last(C.cast(buf, C.c_void_p), C.cast(cnt, C.c_void_p)) == 0:
                acc = [a + b for a, b in zip(acc, buf)]
                nl = list(cnt)
        L.bl_hybrid_timing(0)
        stage_ms = dict(zip(names, [max_over_ranks(v / reps) for v in acc]))
        stage_launches = dict(zip(names, nl))
        hh = shape_d
        regime_counts = {"saddle_point": int(((hh > 13) & (hh <= 170)).sum().item()),
                         "normal": int((hh > 170).sum().item()),
                         "alternate": int(((hh > 1) & (hh <= 13) & (hh != 2)).sum().item()),
                         "devroye": int(((hh == 1) | (hh == 2)).sum().item()),
                         "sum_of_gammas": int(((hh > 0) & (hh < 1)).sum().item())}

    # ---- end to end through the reference-facing C ABI, pinned host buffers ------------
    e2e = None
    if not args.no_e2e:
        shape_p = torch.from_numpy(shape_h).pin_memory()
        z_p = torch.from_numpy(z_h).pin_memory()
        x_p = torch.empty(num, dtype=torch.float64).pin_memory()
        import ctypes as C
        fn_host = L.bl_rpg_hybrid_seeded if wl == "hybrid" else L.bl_rpg_devroye_seeded
        e_steps = max(2, min(args.steps, 3))
        for w in range(2):
            _lib.check(fn_host(x_p.data_ptr(), shape_p.data_ptr(), z_p.data_ptr(), num, SEED, 2000 + w, obs0))
        barrier()
        t0 = time.perf_counter()
        for k in range(e_steps):
            _lib.check(fn_host(x_p.data_ptr(), shape_p.data_ptr(), z_p.data_ptr(), num, SEED, k, obs0))
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        # the host copy must equal the device-resident result of the same stream identity
        step_dev(0)
        torch.cuda.synchronize()
        fn_host(x_p.data_ptr(), shape_p.data_ptr(), z_p.data_ptr(), num, SEED, 0, obs0)
        same = bool(torch.equal(x_p[: 1 << 20], x_d[: 1 << 20].cpu()))
        # the floor under e2e: pinned host->device bandwidth of this rank's link while the
        # device->host direction is busy too, measured now (16 of the 24 bytes per draw go in, 8 come
        # back; the pipeline keeps both directions busy, which costs each ~10 % of its solo rate)
        probe = torch.empty(1 << 26, dtype=torch.float64).pin_memory()
        probe_o = torch.empty(1 << 25, dtype=torch.float64).pin_memory()
        probe_d = torch.empty(1 << 26, dtype=torch.float64, device=dev)
        probe_do = torch.empty(1 << 25, dtype=torch.float64, device=dev)
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

        def both():
            with torch.cuda.stream(s_in):
                probe_d.copy_(probe, non_blocking=True)
            with torch.cuda.stream(s_out):
                probe_o.copy_(probe_do, non_blocking=True)

        both()
        torch.cuda.synchronize()
        tp0 = time.perf_counter()
        for _ in range(3):
            both()
        torch.cuda.synchronize()
        h2d_gbs = 3 * probe.numel() * 8 / (time.perf_counter() - tp0) / 1e9
        del probe, probe_d, probe_o, probe_do
        # the same call with PAGEABLE caller buffers -- what R's .C() hands over (LogitWrapper.R:29,49): the library stages
        # the chunks through its own pinned ring with a pool of copy threads; and, for reference, with that switched
        # off (the driver's own single-threaded staging)
        x_pg = np.zeros(num)
        pageable = {}
        for label, env in (("staged_by_library", None), ("driver_staging", "1")):
            if env:
                os.environ["BAYESLOGIT_NO_STAGING"] = env
            else:
                os.environ.pop("BAYESLOGIT_NO_STAGING", None)
            _lib.check(fn_host(x_pg.ctypes.data, shape_h.ctypes.data, z_h.ctypes.data, num, SEED, 2100, obs0))
            barrier()
            tq = time.perf_counter()
            for k in range(2):
                _lib.check(fn_host(x_pg.ctypes.data, shape_h.ctypes.data, z_h.ctypes.data, num, SEED, k, obs0))
            pageable[label] = world * num * 2 / max_over_ranks(time.perf_counter() - tq)
        os.environ.pop("BAYESLOGIT_NO_STAGING", None)
        fn_host(x_pg.ctypes.data, shape_h.ctypes.data, z_h.ctypes.data, num, SEED, 0, obs0)
        same_pg = bool(np.array_equal(x_pg[: 1 << 20], x_p[: 1 << 20].numpy()))
        del x_pg
        e2e = {"value": world * num * e_steps / dt, "unit": "draws/s", "host_memory": "pinned",
               "rank0_numa_node": numa_node,
               "pageable": {"value": pageable["staged_by_library"], "unit": "draws/s",
                            "frac_of_pinned": pageable["staged_by_library"] / (world * num * e_steps / dt),
                            "driver_staging_value": pageable["driver_staging"],
                            "how": "numpy (malloc) buffers; chunks staged through the library's pinned ring by its copy threads "
                                   "(capi.cu CopyPool); driver_staging_value: the same call with BAYESLOGIT_NO_STAGING=1",
                            "matches_pinned": same_pg},
               "h2d_GBs_measured_with_d2h_busy": h2d_gbs,
               "pcie_bound_draws_per_s": world * h2d_gbs * 1e9 / (BYTES_PER_DRAW[wl] - 8),
               "h2d_bytes_per_step": int(world * num * (BYTES_PER_DRAW[wl] - 8)),
               "d2h_bytes_per_step": int(world * num * 8), "steps": e_steps,
               "api": "rpg_hybrid C ABI, host pointers (pinned)" if wl == "hybrid" else "rpg_devroye C ABI, host pointers (pinned)",
               "matches_device_resident": same}

    # ---- CPU baseline on rank 0, N = 1 only --------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        sample = min(CPU_SAMPLE[wl], num)
        time_cpu(wl, max(sample // 16, 1), cores)
        dt, kind, _ = time_cpu(wl, sample, cores)
        one = max(sample // 8, 1)
        dt1, _, _ = time_cpu(wl, one, 1)
        cpu = {"value": sample / dt, "unit": "draws/s", "cores": cores, "kind": kind,
               "sample": f"first {sample} draws of the workload, all {cores} host threads, {dt:.2f} s wall",
               "value_1_core": one / dt1,
               "sample_1_core": f"first {one} draws of the workload, one thread (the reference's shipped serial loop, "
                                f"LogitWrapper.cpp:129-167), {dt1:.2f} s wall"}

    # ---- extras: the two other figures BASELINE.json's metric names -------------------------
    extras = {}
    if not args.no_extras:
        # (i) PG(1,z) draws/s, z~U(-5,5), 2^27 draws per GPU (north_star target: >= 1e10 on one B200)
        del shape_d, z_d, x_d
        torch.cuda.empty_cache()
        n1 = 1 << 27
        g = torch.Generator(device=dev); g.manual_seed(SEED + rank)
        z1 = torch.rand(n1, generator=g, device=dev, dtype=torch.float64) * 10 - 5
        s1 = torch.ones(n1, device=dev, dtype=torch.int32)
        x1 = torch.empty(n1, device=dev, dtype=torch.float64)
        for w in range(3):
            L.bl_rpg_devroye_dev(x1.data_ptr(), s1.data_ptr(), z1.data_ptr(), n1, SEED, 500 + w, rank * n1, stream)
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for k in range(5):
            L.bl_rpg_devroye_dev(x1.data_ptr(), s1.data_ptr(), z1.data_ptr(), n1, SEED, k, rank * n1, stream)
        b.record()
        barrier()
        ms1 = max_over_ranks(a.elapsed_time(b)) / 5
        extras["pg1"] = {"draws_per_sec": world * n1 / (ms1 * 1e-3), "ms_per_launch": ms1, "draws_per_gpu": n1,
                         "workload": "rpg_devroye PG(1,z), z~U(-5,5), device-resident",
                         "kernel": "k_devroye_refill",
                         "hbm_GBs": n1 * 20 / (ms1 * 1e-3) / 1e9}
        del z1, s1, x1
        torch.cuda.empty_cache()
        # (i') BASELINE config 0 at its stated size: ONE batch of 1M PG(1,z) draws through the drop-in entry with
        # host pointers (what R's .C("rpg_devroye") does), beside the reference's serial loop on one host core
        if rank == 0:
            import numpy as np
            n0 = 1_000_000
            r0 = np.random.default_rng(SEED + 5)
            z0 = r0.uniform(-5.0, 5.0, n0)
            s0 = np.ones(n0, dtype=np.int32)
            x0 = np.empty(n0)
            fn0 = L.bl_rpg_devroye_seeded
            for w in range(3):
                _lib.check(fn0(x0.ctypes.data, s0.ctypes.data, z0.ctypes.data, n0, SEED, 700 + w, 0))
            t0 = time.perf_counter()
            for k in range(10):
                _lib.check(fn0(x0.ctypes.data, s0.ctypes.data, z0.ctypes.data, n0, SEED, k, 0))
            host_ms = (time.perf_counter() - t0) / 10 * 1e3
            c0 = {"batch": n0, "api": "rpg_devroye C ABI, pageable host pointers, one call per batch",
                  "ms_per_batch_e2e": host_ms, "draws_per_sec_e2e": n0 / (host_ms * 1e-3)}
            if not args.no_cpu_baseline:
                O = load_oracle()
                t0 = time.perf_counter()
                O.rpg_devroye(s0, z0, seed=SEED, nthreads=1)
                cpu_s = time.perf_counter() - t0
                c0["cpu_reference_1_core_ms_per_batch"] = cpu_s * 1e3
                c0["cpu_kind"] = O.kind
            extras["config0_pg1_1M_batch"] = c0
        # (ii) logit Gibbs iterations/s at N=1M, P=64 (strong scaling: the N rows are sharded)
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_gibbs
        if world > 1:
            from bayeslogit_b200 import dist as bdist
            bdist.init_comm(rank, world, dev)
        gp = bench_gibbs.run(1_000_000, 64, args.gibbs_iters, 5, False, rank, world, local)
        gc = bench_gibbs.run(1_000_000, 64, max(10, args.gibbs_iters // 10), 2, True, rank, world, local)
        extras["gibbs_logit_N1M_P64"] = {"plain_beta": gp, "reference_constrained_beta": gc, "scaling": "strong"}
        go = bench_gibbs.run(1_000_000, 64, max(20, args.gibbs_iters // 4), 3, False, rank, world, local, one_pass=True)
        extras["gibbs_logit_N1M_P64"]["plain_beta_one_pass_kernel"] = go
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            extras["gibbs_logit_N1M_P64"]["cpu_baseline"] = cpu_gibbs_baseline(1_000_000, 64, 20, 3)
        # (iii) the other sweeps of BASELINE.json's configs: NB regression (config 4), multinomial logit and the
        # batch of independent chains (config 5); short runs, figures per iteration
        import bench_chains
        import bench_models
        torch.cuda.empty_cache()
        extras["chains_4096_N10k_P32"] = bench_chains.run(4096, 10_000, 32, 10, False, rank, world, local, serial_sample=4)
        torch.cuda.empty_cache()
        extras["mlogit_J10_N1M_P32"] = bench_models.run_mlogit(1_000_000, 32, 10, 10, rank, world, local)
        torch.cuda.empty_cache()
        extras["nb_N10M_P256"] = bench_models.run_nb(10_000_000, 256, 6, rank, world, local)
        torch.cuda.empty_cache()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        counters = {}
        try:
            counters = json.load(open(os.path.join(ROOT, "profiles", "ncu_counters.json")))
        except OSError:
            pass
        if stage_ms:
            # dominant kernel = the larger of the two saddle-point kernels (set-up, rejection loop);
            # a step launches it once per state chunk: figures are per launch, averaged over the
            # non-empty launches of the timed pass
            dom_stage = "sp_setup" if stage_ms["sp_setup"] >= stage_ms["sp_loop"] else "sp_loop"
            dom_name = {"sp_setup": "k_sp_setup", "sp_loop": "k_loop_regroup<SpRegroup>"}[dom_stage]
            n_launch = max(1, stage_launches[dom_stage])
            dom_units, dom_ms = regime_counts["saddle_point"] / n_launch, stage_ms[dom_stage] / n_launch
            dom_share = stage_ms[dom_stage] / (total_ms / args.steps)
            # HBM bytes the design moves per saddle-point draw in this kernel (DESIGN.md section 6):
            # set-up: idx 4 + h 8 + z 8 in, 19 state doubles out; loop: idx 4 + h 8 + z 8 + state in, x 8 out
            design_bytes = {"sp_setup": 20 + 152, "sp_loop": 20 + 152 + 8}[dom_stage]
        else:
            dom_units, dom_ms, dom_name = num, kern_ms, "k_devroye_refill"
            dom_share, n_launch, design_bytes = 1.0, 1, BYTES_PER_DRAW[wl]
        hbm_achieved = dom_units * BYTES_PER_DRAW[wl] / (dom_ms * 1e-3) / 1e9
        ctr = counters.get(dom_name, {})
        traffic = None
        if ctr.get("dram_bytes_per_unit") is not None:
            traffic = ctr["dram_bytes_per_unit"] * dom_units
        # The binding roof.  The sampler kernels move 24 B per draw (3 % of HBM at this rate) and are bound by the
        # SM: what they run out of is issue slots (warp instructions per second), so that is the roof quoted --
        # achieved = the warp instructions the kernel EXECUTES per draw (ncu smsp__inst_executed.sum of the same
        # kernel at bench size, profiles/ncu_counters.json) x draws per launch / its live CUDA-event time; peak =
        # the issue rate measured on this device in this run.  The per-pipe shares (ncu pct of peak) follow.
        issue_peak = pipe_peaks["issue_gwarp_inst"]
        if ctr.get("warp_instr_per_unit"):
            issue_achieved = ctr["warp_instr_per_unit"] * dom_units / (dom_ms * 1e-3) / 1e9
            roofline = {"bound": "issue", "achieved": issue_achieved, "peak": issue_peak, "unit": "Gwarp-inst/s",
                        "frac": issue_achieved / issue_peak, "traffic": traffic, "peak_source": "measured (bl_probe_peaks, this run)",
                        "warp_inst_per_unit": ctr["warp_instr_per_unit"],
                        "active_threads_per_warp_inst": ctr.get("active_threads_per_warp_instr"),
                        "pipes_pct_of_peak_ncu": {k: ctr.get(k) for k in ("issue_slots_busy_pct", "fp64_pipe_pct", "fma_pipe_pct",
                                                                            "alu_pipe_pct", "xu_pipe_pct", "lsu_pipe_pct")},
                        "counters_source": ctr.get("source")}
        else:
            roofline = {"bound": "hbm", "achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s",
                        "frac": hbm_achieved / hbm_peak, "traffic": traffic,
                        "peak_source": "measured" if peaks else "fallback",
                        "note": "no ncu instruction counts for this kernel in profiles/ncu_counters.json: HBM roof quoted, "
                                "which does not bind (the sampler is issue-bound)"}
        roofline.update({
            "kernel": dom_name, "kernel_ms": dom_ms, "launches_per_step": n_launch, "units_per_launch": dom_units,
            "share_of_step": dom_share, "stage_ms": stage_ms, "stage_launches": stage_launches, "regime_counts": regime_counts,
            "hbm": {"achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_achieved / hbm_peak,
                    "bytes_per_unit": BYTES_PER_DRAW[wl], "design_bytes_per_unit": design_bytes,
                    "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback",
                    "note": "algorithmic bytes (shape, z in; omega out) against the copy bandwidth: not the binding roof"},
        })
        # the PG(1,z) kernel of the extras against the same issue roof
        if "pg1" in extras and counters.get("k_devroye_refill", {}).get("warp_instr_per_unit"):
            c1 = counters["k_devroye_refill"]
            rate = extras["pg1"]["draws_per_sec"] / world * c1["warp_instr_per_unit"] / 1e9
            extras["pg1"]["roofline"] = {"bound": "issue", "achieved": rate, "peak": issue_peak, "unit": "Gwarp-inst/s",
                                         "frac": rate / issue_peak, "warp_inst_per_unit": c1["warp_instr_per_unit"],
                                         "active_threads_per_warp_inst": c1.get("active_threads_per_warp_instr"),
                                         "counters_source": c1.get("source")}
        out = {
            "metric": "pg_draws_per_sec", "value": value, "unit": "draws/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_config(args),
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "roofline": roofline,
            "peaks_measured": dict(pipe_peaks, hbm_gbs=peaks.get("hbm_gbs"), bf16_tflops=peaks.get("bf16_tflops"),
                                   hbm_source="MEASURED_PEAKS.json (driver-written)" if peaks else "absent"),
            "cpu_baseline": cpu, "mean_omega_first_1M": mean_omega, "extras": extras,
        }
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
