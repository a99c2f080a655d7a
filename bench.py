#!/usr/bin/env python
"""bench.py -- batched NMPC solves/sec (BASELINE.json metric) on N B200s of one node.

One "step" = one pass of the hot path over one batch of synthetic scenes:
solve every scene of the workload once (PANOC + ALM to the reference's tolerances).
The K timed steps rotate through 4 distinct input batches (more bytes than L2 holds) with up
to --depth of them in flight, each on its own stream (DESIGN.md section 3.7): `value` is
scenes / time of all K steps, every step complete inside the timed region.  `sequential`
repeats the steps one batch at a time (the latency of one batch).  `e2e` is the same through
BatchSolver.run_many with pinned host buffers (H2D of the parameters and D2H of every result
field inside the timed region).

  python bench.py --gpus 1 --steps 5 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...      (CPU arm: the oracle on the host cores)
  python bench.py ... --dump-outputs DIR    (results of the last timed step as DIR/<name>.npy)

Prints ONE JSON line (rank 0).  Keys: see the contract in the task; extra objects
`roofline` (FP64 FMA pipe of the solve kernel, peak measured live by a DFMA probe)
and `cpu_baseline` (oracle port on the host cores, bounded sample).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# FP64 floating-point operations per evaluation of the solve kernel, counted from
# csrc/ttmpc_device.cuh for the default shapes (N=20 steps, 10 other robots, 10
# static obstacles x 4 edges, 15 dynamic slots); fma = 2 flops.  See DESIGN.md §kernels.
def eval_flops(cfg, grad: bool, bodies_per_eval: float) -> float:
    N, No, Ns, ne, Nd = cfg.N_hor, cfg.Nother, cfg.Nstcobs, cfg.nstcobs // 3, cfg.Ndynobs
    per_lane = 0.0
    per_lane += 3 * 34 + 14            # three tt_sincos + rollout combination
    per_lane += (N + 1) / 2 * 15       # reference path: avg (N+1)/2 segments x 15 flops
    per_lane += 10                     # speed / control terms
    per_lane += No * 6                 # fleet: distance test
    per_lane += Ns * (ne * 6 + 1)      # static: edges + product
    per_lane += Nd * 5                 # dynamic: bounding test
    per_lane += 22                     # accelerations + ALM rows
    if grad:
        per_lane += 20 + 40            # selected-segment gradient, adjoint combination
    total = per_lane * N
    total += 3 * 5 * 32 + 3 * 5 * 32   # wsum3 + three prefix scans (adds on 32 lanes)
    if grad:
        total += 3 * 5 * 32            # three suffix scans
    total += bodies_per_eval * (34 if grad else 22)
    total += Nd * 4
    return total


def clocks_sampler(stop, out, gpu_index):
    """Sample SM clock, power and throttle reasons during the timed region: NVML every 10 ms when
    pynvml is importable, else nvidia-smi (the recipe's clocks line) every 200 ms."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(gpu_index)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
        while not stop.is_set():
            r = get_reasons(h)
            act = lambda k: "Active" if (r & bits[k]) else "Not Active"
            out.append([str(gpu_index), str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(mx),
                        str(nv.nvmlDeviceGetPowerUsage(h) / 1000.0), hex(r), act("hw_slowdown"),
                        act("hw_thermal_slowdown"), act("sw_thermal_slowdown"), act("sw_power_cap")])
            stop.wait(0.01)
        return
    except Exception:
        pass
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                "-i", str(gpu_index)], capture_output=True, text=True, timeout=5)
            f = [x.strip() for x in r.stdout.strip().split(",")]
            if len(f) >= 9:
                out.append(f)
        except Exception:
            pass
        stop.wait(0.2)


DUMP_FIELDS = ("u", "y", "cost", "exit_status", "outer", "inner", "fpr", "f1", "f2", "pen", "pred")
DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(bufs, out_dir):
    """Write the results of one device solve (the buffers run_device filled) as out_dir/<name>.npy in
    float64, rows in batch order.  `evals` is left out: two of its columns are clock readings.  A batch
    larger than 64 MB is cut to a fixed, seeded sample of scenes; scene_index.npy lists the rows kept."""
    host = {k: bufs[k].double().cpu().numpy() for k in DUMP_FIELDS if bufs[k] is not None}
    n = len(host["cost"])
    per_scene = sum(a[0].nbytes for a in host.values()) + 8
    keep = min(n, DUMP_LIMIT_BYTES // per_scene)
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    host["scene_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a if k == "scene_index" else a[idx])


def summarize_clocks(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no_samples"]}
    sm = sorted(float(s[1]) for s in samples)
    reasons = set()
    for s in samples:
        for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[5:9]):
            if v.lower().startswith("active"):
                reasons.add(name)
    return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(samples[0][2]),
            "power_w_max": max(float(s[3]) for s in samples), "reasons": sorted(reasons),
            "samples": len(samples)}


def parse_workload(name):
    """A named workload of scenes.WORKLOADS, or a sweep shape of BASELINE configs[4]:
    `sweep:N=10,Nstc=10,Ndyn=15` (4096 scenes, 4 static + 3 dynamic obstacles active, default limits)."""
    import trajtrack_mpcndqn_rlboost_b200 as t
    if name.startswith("sweep:"):
        kv = dict(x.split("=") for x in name[6:].split(","))
        N, nst, ndy = int(kv.get("N", 20)), int(kv.get("Nstc", 10)), int(kv.get("Ndyn", 15))
        mc = t.Configurator(N_hor=N, Nstcobs=nst, Ndynobs=ndy)
        w = dict(n=int(kv.get("n", 4096)), n_static=min(4, nst), n_dynamic=min(3, ndy), blocking_fraction=0.1, solver={})
        return mc, mc.to_ttmpc(), w
    w = t.scenes.WORKLOADS[name]
    mc = t.Configurator()
    return mc, mc.to_ttmpc(**w["solver"]), w


def build_workload(name, rank, world, batch=0):
    import trajtrack_mpcndqn_rlboost_b200 as t
    mc, cfg, w = parse_workload(name)
    # weak scaling: every rank solves n scenes per step.  The R distinct input batches are the SAME
    # seeded batches on every rank (seed 1000 + 100 * batch); rank r starts its rotation at batch r
    # (see main), so over K steps (K a multiple of R) the ranks carry exactly equal work and the
    # max-over-ranks time measures the GPUs, not the luck of a rank's seeds.
    p = t.scenes.make_scenes(w["n"], cfg, seed=1000 + 100 * batch, n_static=w["n_static"],
                             n_dynamic=w["n_dynamic"], blocking_fraction=w["blocking_fraction"], mpc=mc)
    return cfg, p, w


def common_config(args, cfg, w, n):
    """The `config` object: identical keys and values in both arms (ours / reference)."""
    return {"workload": args.workload, "scenes_per_step_per_gpu": int(w["n"]), "N_hor": cfg.N_hor,
            "Nother": cfg.Nother, "Nstcobs": cfg.Nstcobs, "Ndynobs": cfg.Ndynobs,
            "static_per_scene": w["n_static"], "dynamic_per_scene": w["n_dynamic"],
            "max_inner": cfg.max_inner_iterations, "max_outer": cfg.max_outer_iterations,
            "iteration_limits": ("opengen 0.7.1 defaults (500 x 10)" if cfg.max_inner_iterations == 500 else
                                 "ASSUMPTION: config/mpc_longiter.yaml differs from mpc_default.yaml only in "
                                 "optimizer_name; 2000 x 20 taken as its 'long iteration' limits (DESIGN.md section 6)"),
            "distinct_batches": max(1, args.batches),
            "inputs": "seeded synthetic scenes (scenes.make_scenes, seeds 1000 + 100 j), the same batches on every rank"}


def run_reference_arm(args):
    """CPU arm: the oracle (port of the OpEn solve, reference operation order) on all
    host cores, on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from tests import oracle_lib as O
    R = max(1, args.batches)
    cfg, p0, w = build_workload(args.workload, 0, 1, 0)
    ps = [p0] + [build_workload(args.workload, 0, 1, j)[1] for j in range(1, R)]  # the batches the GPU arm rotates through
    cores = os.cpu_count() or 1
    sample = min(len(p0), args.cpu_sample)
    O.load()
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        O.solve_batch(cfg, ps[it % R][:sample], threads=cores, warp=False)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = sample * len(times) / total
    line = {
        "impl": "reference", "metric": "batched NMPC solves/sec", "value": value, "unit": "solves/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": common_config(args, cfg, w, sample),
        "run_info": {"scenes_per_step": sample,
                     "note": "OpEn is Rust and absent here: CPU port (oracle, reference operation "
                             "order) on all host cores; each step = a bounded sample of the workload"},
        "cpu_baseline": {"value": value, "unit": "solves/s", "cores": cores, "kind": "port",
                         "sample": f"first {sample} scenes of each of the {R} rotating {args.workload} batches, pthreads"},
        "e2e": {"value": value, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="static4096")
    ap.add_argument("--cpu-sample", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--depth", type=int, default=0,
                    help="batches in flight (1 = one at a time; 0 = auto: the divisor of --steps closest to 6 in 4..8, "
                         "so that every stream carries the same number of steps and the region does not end with one or two streams still busy)")
    ap.add_argument("--batches", type=int, default=4, help="distinct input batches the steps rotate through")
    ap.add_argument("--e2e-depth", type=int, default=0,
                    help="host calls in flight in the e2e leg (0 = the same number as --depth; measured on one B200 with "
                         "20 steps, tools/e2e_ab.py: 5 calls 552 k, 6 calls 537 k, 7 calls 530 k, 8 calls 527 k solves/s)")
    ap.add_argument("--quick", action="store_true", help="sweep rows: skip the sequential / pageable / one-scene legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step (rank 0) as DIR/<name>.npy, float64, at most "
                         "64 MB (a fixed, seeded sample of scenes beyond that): two builds run with the same "
                         "arguments solve the same inputs and can be compared output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    import trajtrack_mpcndqn_rlboost_b200 as t
    from trajtrack_mpcndqn_rlboost_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the solver has no CPU path")
    # host threads this rank may use for staging pageable inputs: its share of half the cores
    os.environ.setdefault("TTMPC_HOST_THREADS", str(max(1, (os.cpu_count() or 1) // (2 * max(1, world)))))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # R distinct input batches rotate through the steps: 4 x 87 MB of parameters > 126 MB of L2, so
    # no step finds its inputs in L2 (the one-batch-at-a-time leg flushes L2 explicitly as well)
    R = max(1, args.batches)
    cfg, p0, w = build_workload(args.workload, rank, world, 0)
    p_hosts = [p0] + [build_workload(args.workload, rank, world, j)[1] for j in range(1, R)]
    p_host = p_hosts[0]
    n = len(p_host)
    solver = t.BatchSolver(cfg)
    lib = _lib.load()
    dev = torch.device("cuda", local)
    p_devs = [torch.from_numpy(p).pin_memory().to(dev, non_blocking=True) for p in p_hosts]
    if args.depth <= 0:  # equal number of steps per stream: 20 steps -> 5 streams x 4 (6 streams would leave 2 of them a 4th step)
        cand = [d for d in (6, 5, 7, 8, 4) if args.steps % d == 0]
        args.depth = cand[0] if cand else 6
    D = max(1, args.depth)
    bufs_ring = [solver.alloc_device(n, device=dev) for _ in range(D)]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # 256 MB > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        tns = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(tns, op=dist.ReduceOp.MAX)
        return float(tns.item())

    def gather_ranks(vals):
        """[world][len(vals)] float64 over NCCL (results and metrics are what NCCL is for here:
        there is no collective in the solve)."""
        tns = torch.tensor(list(vals), dtype=torch.float64, device=dev)
        if world == 1:
            return tns[None, :].cpu().numpy()
        out = [torch.empty_like(tns) for _ in range(world)]
        dist.all_gather(out, tns)
        return torch.stack(out).cpu().numpy()

    rot = rank % R  # this rank's first batch of the rotation (equal work on every rank, see build_workload)

    main_stream = torch.cuda.current_stream()
    # ---------------- one batch at a time ("sequential"): per-batch latency.  Each step is timed by
    # its own event pair, L2 flushed before it; the next step starts when this one has ended.
    seq_ms = []
    seq_steps = 2 if args.quick else args.steps
    for it in range(args.warmup + seq_steps):
        if it == args.warmup:
            barrier()
        flush.zero_()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(main_stream)
        solver.run_device(p_devs[(it + rot) % R], bufs_ring[0])
        e1.record(main_stream)
        if it >= args.warmup:
            seq_ms.append((e0, e1))
    barrier()
    seq_ms = [a.elapsed_time(b) for a, b in seq_ms]
    seq_step_ms = max_over_ranks(sum(seq_ms) / len(seq_ms))
    # ---------------- device-resident leg ("value"): the same K steps with up to D batches in
    # flight.  Step i runs on stream i mod D with its own output buffers; the library gives each
    # stream its own scene queue, so the CTAs of the next batch become resident as the CTAs of
    # the running one drain and its tail (a few long scenes on an otherwise idle GPU) is filled.
    # Timed by ONE event pair around all K steps, every step complete at the second event.
    streams = [torch.cuda.Stream(device=dev) for _ in range(D)]

    done_ev = {}

    def issue(first, count, mark=False):
        for it in range(first, first + count):
            with torch.cuda.stream(streams[it % D]):
                solver.run_device(p_devs[(it + rot) % R], bufs_ring[it % D])
                if mark:  # completion time of every step: the drain of the region is read from these
                    done_ev[it] = torch.cuda.Event(enable_timing=True)
                    done_ev[it].record(streams[it % D])

    def fork():
        for s_ in streams:
            s_.wait_stream(main_stream)

    def join():
        for s_ in streams:
            main_stream.wait_stream(s_)

    warm = max(args.warmup, D)  # every stream's scene queue and scratch tables exist before the timed region
    fork(); issue(0, warm); join()
    barrier()
    solver.read_stats(reset=True)
    samples, stop = [], threading.Event()
    th = threading.Thread(target=clocks_sampler, args=(stop, samples, local), daemon=True)
    th.start()
    t_wall0 = time.perf_counter()
    ev_a = torch.cuda.Event(enable_timing=True); ev_b = torch.cuda.Event(enable_timing=True)
    ev_a.record(main_stream)
    fork(); issue(warm, args.steps, mark=True); join()
    ev_b.record(main_stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    stop.set()
    if args.dump_outputs and rank == 0:  # before the buffers are reused below
        dump_outputs(bufs_ring[(warm + args.steps - 1) % D], args.dump_outputs)
    total_ms = ev_a.elapsed_time(ev_b)
    stats = solver.read_stats(reset=True)
    local_ms = total_ms / args.steps
    step_ms = max_over_ranks(local_ms)
    total_scenes = n * world
    value = total_scenes / (step_ms * 1e-3)
    # when did each step complete?  drain = the end of the region during which fewer than D batches
    # are in flight (from the completion of step K - D to the end), the part a longer run amortises
    done_t = sorted(ev_a.elapsed_time(done_ev[it]) for it in done_ev)
    drain_ms = total_ms - (done_t[-D] if len(done_t) >= D else 0.0)
    # exit status of every distinct batch, for the cross-check against the host path below
    status = []
    for j in range(R):
        solver.run_device(p_devs[j], bufs_ring[0]); torch.cuda.synchronize()
        status.append(bufs_ring[0]["exit_status"].cpu().numpy().copy())
    # results and metrics of every rank, gathered over NCCL
    steps_per_batch = [sum(1 for it in range(warm, warm + args.steps) if (it + rot) % R == j) for j in range(R)]
    hist_local = sum(np.bincount(status[j], minlength=4) * steps_per_batch[j] for j in range(R))
    per_rank = gather_ranks([local_ms, drain_ms, stats["cost_evals"], stats["grad_evals"], stats["panoc_iters"],
                             stats["dyn_bodies"], *hist_local.tolist()])

    # ---------------- end-to-end leg ("e2e"): the reference-facing call with HOST buffers,
    # BatchSolver.run -> ttmpc_solve_batch_host: host parameters -> pinned staging -> H2D,
    # solve, D2H of every result field, all inside the timed region; K calls, up to D in flight
    # (BatchSolver.run_many: one host thread per in-flight call).
    # Inputs sit in pinned host memory (numpy views of pinned torch tensors): the library copies from
    # them directly.  The same calls on pageable numpy arrays (staged through the library's pinned
    # buffer by a host memcpy first) are reported as e2e.pageable_value.
    p_pins = []
    for p in p_hosts:
        pp = t.pinned_empty(p.shape)
        pp[...] = p
        p_pins.append(pp)

    def e2e_leg(arrays, depth, steps):
        host_steps = [arrays[(it + rot) % R] for it in range(steps)]
        solver.run_many(host_steps[:max(2, depth)], depth=depth)
        barrier()
        t0 = time.perf_counter()
        sols = solver.run_many(host_steps, depth=depth)
        dt = time.perf_counter() - t0
        for it, hs in enumerate(sols):
            assert np.array_equal(hs.exit_status, status[(it + rot) % R]), "host and device paths disagree"
        return max_over_ranks(dt / steps)

    DE = max(1, min(8, args.e2e_depth if args.e2e_depth > 0 else D))
    e2e_step = e2e_leg(p_pins, DE, args.steps)
    e2e_value = total_scenes / e2e_step
    if args.quick:
        e2e_pageable_step = e2e_seq_step = float("nan")
    else:
        e2e_pageable_step = e2e_leg(p_hosts, DE, args.steps)
        # one call at a time (latency of the blocking call)
        e2e_seq_step = e2e_leg(p_pins, 1, min(args.steps, 8))
    h2d = p_host.nbytes
    N = cfg.N_hor
    d2h = n * (2 * 2 * N * 8 + 5 * 8 + N * 3 * 8 + 3 * 4 + 4 * 8)
    exit_hist = per_rank[:, 6:10].sum(axis=0).astype(np.int64).tolist()  # whole job, timed region

    # ---------------- roofline of the solve kernel: FP64 FMA pipe
    peak = C.c_double()
    _lib.check(lib.ttmpc_measure_fp64_peak(C.byref(peak), None), "fp64 peak probe")
    steps = args.steps
    n_cost = stats["cost_evals"] / steps
    n_grad = stats["grad_evals"] / steps
    bodies = stats["dyn_bodies"] / max(1.0, (stats["cost_evals"] + stats["grad_evals"]))
    flops = n_cost * eval_flops(cfg, False, bodies) + n_grad * eval_flops(cfg, True, bodies)
    achieved = flops / (local_ms * 1e-3) / 1e12
    # DRAM traffic and EXECUTED fp64 instructions of one launch come from the tracked ncu summary of
    # the same kernel on the same workload (profiles/r2_roofline_inputs.json names its source file):
    # executed flops per evaluation x the evaluations of THIS run = executed flop rate, next to the
    # algorithmic one (which counts the reference expression, zero-padded slots included).
    prof = {}
    try:
        with open(os.path.join(ROOT, "profiles", "r2_roofline_inputs.json")) as f:
            prof = json.load(f).get(args.workload, {})
    except Exception:
        prof = {}
    executed = None
    if prof.get("executed_flops_per_eval"):
        executed = prof["executed_flops_per_eval"] * (n_cost + n_grad) / (local_ms * 1e-3) / 1e12
    roofline = {"bound": "fp64_fma", "achieved": achieved, "peak": peak.value, "unit": "TFLOP/s",
                "frac": achieved / peak.value if peak.value else None,
                "traffic": prof.get("dram_bytes_per_launch"),
                "traffic_source": prof.get("source"),
                "algorithmic_bytes_per_launch": int(p_host.nbytes + d2h),
                "executed_TFLOPs": executed,
                "executed_frac": executed / peak.value if (executed and peak.value) else None,
                "executed_flops_per_eval": prof.get("executed_flops_per_eval"),
                "algorithmic_flops_per_eval": flops / max(1.0, n_cost + n_grad),
                "peak_source": "measured live: DFMA probe kernel (ttmpc_measure_fp64_peak); "
                               "MEASURED_PEAKS.json has no FP64 entry",
                "hbm_GBps_algorithmic": (p_host.nbytes + d2h) / (local_ms * 1e-3) / 1e9,
                "evals_per_solve": (n_cost + n_grad) / n,
                "panoc_iters_per_solve": stats["panoc_iters"] / steps / n}

    # ---------------- CPU baseline (rank 0, N=1 only): oracle port on the host cores
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from tests import oracle_lib as O
        cores = os.cpu_count() or 1
        sample = min(n, args.cpu_sample)
        O.load()
        t0 = time.perf_counter()
        O.solve_batch(cfg, p_host[:sample], threads=cores, warp=False)
        dt = time.perf_counter() - t0
        cpu = {"value": sample / dt, "unit": "solves/s", "cores": cores, "kind": "port",
               "sample": f"first {sample} scenes of {args.workload}, {dt:.1f} s, pthreads"}

    # ---------------- plan latency (the second half of BASELINE's metric): one scene per call on the
    # device (the drop-in Solver.run use), next to the latency of one whole batch measured above
    latency = {"batch_of_%d_ms" % n: seq_step_ms}
    try:
        one = solver.alloc_device(1, device=dev)
        ts = []
        for i in range(0 if args.quick else 48):
            a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
            a.record(main_stream)
            solver.run_device(p_devs[0][i:i + 1], one)
            b.record(main_stream)
            torch.cuda.synchronize()
            if i >= 8:
                ts.append(a.elapsed_time(b))
        ts.sort()
        if ts:
            latency.update({"one_scene_p50_ms": ts[len(ts) // 2], "one_scene_max_ms": ts[-1], "one_scene_samples": len(ts)})
    except Exception as e:  # a diagnostic must never cost the bench line
        latency["one_scene_error"] = repr(e)

    if rank == 0:
        info = solver.launch_info(n)
        line = {
            "metric": "batched NMPC solves/sec", "value": value, "unit": "solves/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": common_config(args, cfg, w, n),
            "run_info": {"pipeline_depth": D, "warmup_steps_run": warm,
                         "l2": f"{R} distinct resident batches of {p_host.nbytes / 1e6:.0f} MB rotate through the steps "
                               f"({R * p_host.nbytes / 1e6:.0f} MB > 126 MB L2): no step finds its inputs in L2",
                         "timing": "one CUDA-event pair around all K steps (up to pipeline_depth batches in flight, "
                                   "each on its own stream, all complete at the second event); 'sequential' = one "
                                   "batch at a time, an event pair per step, L2 flushed by a 256 MB write before each",
                         "parallelism": f"scenes sharded, {world} rank(s), no collective in the solve; NCCL gathers "
                                        "the per-rank times, counters and exit-status histograms",
                         "launch": info},
            # every rank's own device time per step and the drain at the end of its timed region
            "per_rank": {"ms_per_step": [round(x, 4) for x in per_rank[:, 0].tolist()],
                         "ms_per_step_min_mean_max": [float(per_rank[:, 0].min()), float(per_rank[:, 0].mean()),
                                                      float(per_rank[:, 0].max())],
                         "drain_ms": [round(x, 3) for x in per_rank[:, 1].tolist()],
                         "evals_per_step": [float(x) for x in ((per_rank[:, 2] + per_rank[:, 3]) / args.steps).tolist()],
                         "exit_status_hist": per_rank[:, 6:10].astype(np.int64).tolist()},
            # one batch at a time: what a caller that waits for each batch before sending the next sees
            "sequential": {"value": total_scenes / (seq_step_ms * 1e-3), "ms_per_step": seq_step_ms,
                           "e2e_value": total_scenes / e2e_seq_step, "e2e_ms_per_step": e2e_seq_step * 1e3},
            "e2e": {"value": e2e_value, "unit": "solves/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_step * 1e3,
                    "calls_in_flight": DE, "inputs": "pinned host memory",
                    "pageable_value": total_scenes / e2e_pageable_step},
            # per step: solve_kernel, plus rank_scenes_kernel + order_scenes_kernel when the batch
            # is larger than the resident warps (dispatch order)
            "gpu_launches": args.steps * (3 if n > info["grid"] * info["block"] // 32 else 1),
            "plan_latency": latency,
            "clocks": summarize_clocks(samples),
            "roofline": roofline,
            "cpu_baseline": cpu,
            "exit_status_hist": exit_hist,
            "wall_s_timed_region": t_wall,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
