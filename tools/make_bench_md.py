#!/usr/bin/env python
"""BENCH.md (round 2) from the measurement files the tools leave in gpurun_out/:
r2_bench_static4096.json (headline), r2_bench_reference.json, r2_multi_<tag>_n<N>.json (tools/r2_multi.sh,
tools/r2_single_sweep.sh), profiles/r2_parity_distribution_{gpu,cpu}.json, r2_qnet.json, r2_fleet.json,
r2_hybrid.json, r2_single_latency.txt, profiles/r2_roofline_inputs.json, r2_missions.json (tools/bench_missions.py,
one line per fleet size), r2_missions_profile.json (its --profile-pack line), r2_monitor.json (tools/bench_monitor.py),
r2_lidar_moving.json (tools/bench_lidar_moving.py), r2_hybrid_lidar.json (tools/bench_hybrid.py timing runs with and
without --lidar-moving), r2_hybrid_drive.json (its --monitor drives), r2_world.json (tools/bench_world.py)."""
import glob
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "gpurun_out")
P = os.path.join(ROOT, "profiles")


def rd(path):
    return open(path).read() if os.path.exists(path) else ""


def jl(path):
    out = []
    for l in rd(path).splitlines():
        l = l.strip()
        if l.startswith("{"):
            try:
                out.append(json.loads(l))
            except Exception:
                pass
    return out


def last(path):
    x = jl(path)
    return x[-1] if x else None


R1 = {  # round-1 numbers of the same rows (BENCH.md of round 1, one B200)
    "static4096": 436548, "mixed4096": 172285, "dynamic8192": 10917,
    "sweep_N_10_Nstc_10_Ndyn_15": 201758, "sweep_N_32_Nstc_10_Ndyn_15": 70989,
    "sweep_N_20_Nstc_4_Ndyn_4": 125632, "sweep_N_20_Nstc_20_Ndyn_30": 107521,
}


def parity_table(rows):
    out = ["| workload | comparison | exit status agrees | \\|Δu\\| ≤ 1e-4 | \\|Δu\\| p50 / p99 / max | cost within 1e-6 rel. | both converged: \\|Δu\\| ≤ 1e-4, p50 / p99 |",
           "|---|---|---:|---:|---|---:|---|"]
    for name, r in rows.items():
        arm = "GPU" if r.get("kernel_arm") == "gpu" else "kernel order (WARP-order oracle)"
        for key, label in (("kernel_vs_reference_order", f"{arm} vs reference order"),
                           ("reference_order_vs_itself_1ulp", "reference order vs itself, p ± 1 ulp")):
            c = r[key]
            conv = "—"
            if "conv_du_p50" in c:
                conv = f"{100 * c['conv_du_le_1e4']:.1f} %, {c['conv_du_p50']:.1e} / {c['conv_du_p99']:.1e} (n={c['both_converged']})"
            out.append(f"| `{name}` (n={c['n']}) | {label} | {100 * c['status_agree']:.1f} % | {100 * c['du_le_1e4']:.1f} % | "
                       f"{c['du_p50']:.1e} / {c['du_p99']:.1e} / {c['du_max']:.2f} | {100 * c['cost_rel_le_1e6']:.1f} % | {conv} |")
    return out


def missions_section(ms, prof):
    """Lines of the "Missions" table: rows of tools/bench_missions.py, prof: its --profile-pack line."""
    if not ms:
        return []
    out = ["## Missions (`tools/bench_missions.py`; robots take their next task on arrival)\n",
           f"`make_missions(n, {ms[0]['tasks']}, seed=1000)`: a chain of {ms[0]['tasks']} tasks per robot. S / WS: the "
           "queued tasks are taken inside the step (`FleetPlanner.set_tasks`, skip stopped robots, WS also warm "
           "start). H: the same fleet re-tasked from the host after every step (sync, `get_global_ref_traj` per "
           f"arrived robot, copies back); its host time is the time spent in that code, the wait for the step at the sync included. Legs interleaved S WS H H WS S, at most {ms[0]['max_steps']} steps; each row "
           f"is the mean of two legs. {ms[0]['gpu']}, power limit {ms[0]['power_limit']}.\n",
           "| robots | leg | tasks completed | steps | drive time (s) | tasks / s | robot-steps / s | ms / step p50 | p90 | host time (s) |",
           "|---:|:--|---:|---:|---:|---:|---:|---:|---:|---:|"]
    for r in ms:
        for leg, m in r["mean"].items():
            host = f"{m['host_s']:.2f}" if "host_s" in m else "–"
            out.append(f"| {r['robots']} | {leg} | {m['tasks_completed']:,.0f} | {m['steps']:.0f} | {m['drive_s']:.2f} | "
                       f"{m['tasks_per_s']:,.0f} | {m['robot_steps_per_s']:,.0f} | {m['step_ms_p50']:.1f} | {m['step_ms_p90']:.1f} | {host} |")
    out.append("")
    if prof:
        p = prof["profile_pack"]
        out.append(f"`fleet_pack_kernel` with {p['robots']} robots (`--profile-pack`, torch.profiler): {p['all_switch']['pack_us']:.0f} µs "
                   f"in a step in which every robot takes a task ({p['switched_in_first_step']} switched), "
                   f"{p['no_switch']['pack_us']:.0f} µs in the next step, in which none does.\n")
    return out


def monitor_section(mo):
    """Lines of the "Fleet monitor" section: the line of tools/bench_monitor.py."""
    if not mo:
        return []
    out = ["## Fleet monitor (`tools/bench_monitor.py`; swept clearance, contacts and tracking deviation after every step)\n",
           f"Kernel time of `fleet_monitor_kernel` on `make_fleet(n, seed=1000)` geometry (4 rectangles and 2 moving obstacles "
           f"per robot, the chords of the third step), one pair of CUDA events per launch, {mo['gpu']}, power limit {mo['power_limit']}.\n",
           "| robots | launches | µs p50 | µs mean |", "|---:|---:|---:|---:|"]
    for k in mo["kernel"]:
        out.append(f"| {k['robots']} | {k['launches']} | {k['kernel_us_p50']:.1f} | {k['kernel_us_mean']:.1f} |")
    out.append("")
    out.append("One thread per robot: both sizes are a single wave of CTAs (32 and 128 on 148 SMs), so the time is the "
               "latency of one robot's chain of fp64 divisions and square roots, not a throughput.\n")
    d = mo.get("drive")
    if d:
        q = d["min_clearance_quantiles"]
        out.append(f"Drive: `make_fleet({d['robots']}, seed=1000)`, {d['steps']} steps, options {d['options']}, default monitor (robot "
                   f"centre against the polygons the MPC sees, moving obstacles as discs of {d['moving_radius']} m). Reached / failed / "
                   f"running {d['reached']} / {d['failed']} / {d['running']}; robots with contact {d['robots_with_contact']} "
                   f"({d['contact_steps_total']} robot-steps in contact); min_clearance quantiles 0 / 1 / 5 / 10 / 50 %: "
                   + " / ".join(f"{q[k]:.3f}" for k in ("0.0", "0.01", "0.05", "0.1", "0.5"))
                   + f" m; tracking deviation mean {d['deviation_mean']:.3f} m, max {d['deviation_max']:.3f} m.\n")
    s = mo.get("drive_static_only")
    if s:
        q = s["min_clearance_quantiles"]
        out.append(f"The same drive with moving_radius = 0, i.e. the rectangles alone: robots with contact {s['robots_with_contact']} "
                   f"({s['contact_steps_total']} robot-steps); min_clearance quantiles "
                   + " / ".join(f"{q[k]:.3f}" for k in ("0.0", "0.01", "0.05", "0.1", "0.5")) + " m.\n")
    return out


def world_section(lines):
    """Lines of the "Shared obstacle map" section: the lines of tools/bench_world.py."""
    sel = [r for r in lines if r.get("bench") == "world_select"]
    drv = [r for r in lines if r.get("bench") == "world_drive"]
    if not (sel or drv):
        return []
    out = ["## Shared obstacle map (`tools/bench_world.py`; `ttmpc_fleet_world_select_device` before every step)\n"]
    if sel:
        r0 = sel[0]
        out += [f"`make_warehouse(n, tasks=1, seed=1000, shelves=M)` (1 m x 4 m shelves, 3 m aisles: the same density at every M), "
                f"robots at their start crossings, Nstcobs = {r0['nstcobs']}, reach = cell = 6 m; {r0['gpu']}, power limit "
                f"{r0['power_limit']}. Selection: CUDA events over 200 warm launches; step: the whole step (selection + pack + "
                "solve + advance, warm start and skip-stopped), mean of 10 steps after 3.\n",
                "| robots | shelves M | selection ms | step ms | selection / step | world_reach max | mean |",
                "|---:|---:|---:|---:|---:|---:|---:|"]
        for r in sel:
            out.append(f"| {r['robots']} | {r['shelves']:,} | {r['select_ms']:.3f} | {r['step_ms']:.2f} | "
                       f"{100 * r['select_share_of_step']:.1f} % | {r['world_reach_max']} | {r['world_reach_mean']:.2f} |")
        out.append("")
    for d in drv:
        out += [f"Drive: `make_warehouse({d['robots']}, tasks={d['tasks']}, seed=1000)` ({d['shelves']:,} shelves), up to "
                f"{d['max_steps']} steps per leg, legs S WS WS S (skip-stopped, WS also warm start), the monitor on the map "
                f"(robot centre against every shelf); {d['gpu']}, power limit {d['power_limit']}.\n",
                "| leg | steps | tasks completed | step ms p50 | p90 | robots with contact | world_reach max | robot-steps with world_reach > Nstcobs |",
                "|---|---:|---:|---:|---:|---:|---:|---:|"]
        for r in d["legs"]:
            out.append(f"| {r['leg']} | {r['steps']} | {r['tasks_completed']} | {r['step_ms_p50']:.2f} | {r['step_ms_p90']:.2f} | "
                       f"{r['robots_with_contact']} | {r['world_reach_max']} | {r['robot_steps_reach_over_nstcobs']:,} |")
        out.append("")
        out.append("The drive's step time includes the monitor, which measures every robot against every shelf (O(M) per "
                   "robot); the selection table's step time has no monitor.\n")
    return out


def lidar_moving_section(lm, hy, drive):
    """Lines of the "Moving obstacles in the lidar" section: the line of tools/bench_lidar_moving.py, the lines of
    tools/bench_hybrid.py with and without --lidar-moving (hy: timing runs, drive: --monitor runs)."""
    if not (lm or hy or drive):
        return []
    out = ["## Moving obstacles in the DQN's lidar (`ttdqn_observe_act_moving_device`, `--lidar-moving`)\n"]
    if lm:
        m = lm["ms_per_call_median"]
        out.append(f"`tools/bench_lidar_moving.py`, {lm['n_envs']} environments, observation + Q-network per call (median of "
                   f"{lm['rounds']} rounds of {lm['calls']} calls), {lm['gpu']}, power limit {lm['power_limit']}: static rings alone "
                   f"{m['static']:.3f} ms; with 2 moving squares through the new path {m['moving2']:.3f} ms; the same 2 squares "
                   f"appended as static rings {m['appended2']:.3f} ms. Outputs of the last two identical: {lm['moving2_equals_appended2']}.\n")
    if hy:
        rows = {}
        for r in hy:
            rows.setdefault(bool(r.get("lidar_moving")), []).append(r)
        out.append(f"`tools/bench_hybrid.py {hy[0]['envs']} {hy[0]['steps']}` (runs alternated, mean over the runs of each run's per-step p50), "
                   f"{hy[0]['gpu']}, power limit {hy[0]['power_limit']}:\n")
        out += ["| lidar | runs | ms / step p50 | DQN part ms p50 | env-steps / s | hint on |", "|:--|---:|---:|---:|---:|---:|"]
        for mv, rs in sorted(rows.items()):
            med = lambda k: sum(r[k] for r in rs) / len(rs)
            out.append(f"| {'static + moving squares' if mv else 'static only'} | {len(rs)} | {med('step_ms_p50'):.2f} | "
                       f"{med('dqn_part_ms_p50'):.3f} | {med('env_steps_per_s'):,.0f} | {rs[-1]['hint_on']} |")
        out.append("")
    if drive:
        d0 = drive[0]
        out.append(f"Drive: `make_fleet({d0['envs']}, seed=1000)`, {d0['steps'] + 3} steps (3 warm-up + {d0['steps']} timed), warm start + "
                   f"skip-stopped, the default monitor ({d0['gpu']}, power limit {d0['power_limit']}). This is a finding about the planner, "
                   "not a target: whether the trained policy steers better with the extra input was not known before this run.\n")
        out += ["| lidar | reached | running | robots with contact | deepest moving-disc entry (m) | hint on at the end |",
                "|:--|---:|---:|---:|---:|---:|"]
        for r in drive:
            out.append(f"| {'static + moving squares' if r.get('lidar_moving') else 'static only (blind)'} | {r['reached']} | {r['running']} | "
                       f"{r['robots_with_contact']} | {r['deepest_moving_disc_entry']:.3f} | {r['hint_on']} |")
        out.append("")
    return out


def main():
    out = ["# BENCH — round 2 measurements (B200, gpurun; generated by `tools/make_bench_md.py`)\n",
           "Timing with CUDA events on the device; `e2e` = `BatchSolver.run_many` with host numpy buffers; CPU = the oracle in the "
           "reference's operation order on all host cores of the GPU box, bounded sample. Round-1 figures of the same rows are quoted "
           "next to the new ones.\n"]
    b = last(os.path.join(G, "r2_bench_static4096.json"))
    ref = last(os.path.join(G, "r2_bench_reference.json"))
    if b:
        ro, sq, pr = b["roofline"], b.get("sequential", {}), b.get("per_rank", {})
        # the ncu capture of the SAME build is taken after the bench ran: executed flops / DRAM bytes from the current inputs
        ri = json.load(open(os.path.join(P, "r2_roofline_inputs.json"))).get(b["config"]["workload"])
        if ri and ro.get("traffic_source") != ri["source"]:
            evals_per_s = ro["evals_per_solve"] * b["value"]
            ro = dict(ro, traffic=ri["dram_bytes_per_launch"], traffic_source=ri["source"], executed_flops_per_eval=ri["executed_flops_per_eval"],
                      executed_TFLOPs=evals_per_s * ri["executed_flops_per_eval"] / 1e12,
                      executed_frac=evals_per_s * ri["executed_flops_per_eval"] / 1e12 / ro["peak"])
        out.append("## Headline (`python bench.py`, BASELINE `configs[1]`)\n")
        out.append(f"`{b['config']['workload']}`, {b['steps']} steps, {b['run_info']['l2']}, up to {b['run_info']['pipeline_depth']} batches in flight: "
                   f"**{b['value']:,.0f} solves/s** device-resident ({b['ms_per_step']:.2f} ms per 4096-scene step; round 1: 436,548), "
                   f"**{b['e2e']['value']:,.0f} solves/s** end to end from pinned host buffers ({b['e2e']['ms_per_step']:.2f} ms per step; "
                   f"{b['e2e']['h2d_bytes_per_step'] / 1e6:.0f} MB H2D + {b['e2e']['d2h_bytes_per_step'] / 1e6:.1f} MB D2H per step; "
                   f"{b['e2e'].get('pageable_value', 0):,.0f} from pageable arrays; round 1: 408,237). "
                   f"SM clock {b['clocks']['sm_mhz']:.0f} MHz, throttle reasons {b['clocks']['reasons']}.\n")
        out.append(f"Roofline `{ro['bound']}`: {ro['achieved']:.2f} TFLOP/s algorithmic of {ro['peak']:.1f} measured by the DFMA probe = **{100 * ro['frac']:.1f} %** "
                   f"(round 1: 5.8 %)" + (f"; executed fp64 flops (2·DFMA + DADD + DMUL thread instructions from `{ro.get('traffic_source')}`, "
                   f"{ro['executed_flops_per_eval']:,.0f} per evaluation against {ro['algorithmic_flops_per_eval']:,.0f} algorithmic): {ro['executed_TFLOPs']:.2f} TFLOP/s = {100 * ro['executed_frac']:.1f} %"
                   if ro.get("executed_TFLOPs") else "") +
                   (f"; DRAM traffic of one launch {ro['traffic'] / 1e6:.1f} MB against {ro['algorithmic_bytes_per_launch'] / 1e6:.1f} MB algorithmic" if ro.get("traffic") else "") +
                   f"; {ro['evals_per_solve']:.0f} evaluations and {ro['panoc_iters_per_solve']:.0f} PANOC iterations per solve.\n")
        if pr:
            out.append(f"Timed region: {b['ms_per_step'] * b['steps']:.0f} ms for {b['steps']} steps, of which the drain (fewer than "
                       f"{b['run_info']['pipeline_depth']} batches in flight at the end) is {pr['drain_ms'][0]:.0f} ms.\n")
        st = last(os.path.join(P, "r2_bench_lines_100_steps.json"))
        if st:
            a, m = st["static4096_100_steps"], st["mixed4096_100_steps"]
            out.append(f"Steady state — the same command with `--steps 100` (the drain at the end of the timed region weighs five times less): "
                       f"**{a['value']:,.0f} solves/s** device-resident, {a['e2e']['value']:,.0f} end to end; `mixed4096`: {m['value']:,.0f} / {m['e2e']['value']:,.0f} "
                       f"(`profiles/r2_bench_lines_100_steps.json`; measured one step before the shipped build — without the inlined L-BFGS butterflies, "
                       f"662,759 solves/s under the 20-step protocol).\n")
        if sq:
            out.append(f"One batch at a time (L2 flushed before each): {sq['value']:,.0f} solves/s, **{sq['ms_per_step']:.1f} ms per 4096-scene batch** "
                       f"(round 1: 21.5 ms); host call {sq['e2e_ms_per_step']:.1f} ms.\n")
        lat = b.get("plan_latency", {})
        if lat.get("one_scene_p50_ms"):
            out.append(f"One scene per call on the device: p50 {lat['one_scene_p50_ms']:.2f} ms, max {lat['one_scene_max_ms']:.2f} ms (round 1: 1.28 ms p50).\n")
        if b.get("cpu_baseline"):
            c = b["cpu_baseline"]
            out.append(f"CPU port ({c['kind']}): {c['value']:,.0f} solves/s on {c['cores']} cores ({c['sample']}).\n")
    if ref:
        out.append(f"`bench.py --impl reference`: {ref['value']:,.0f} solves/s on {ref['cpu_baseline']['cores']} host cores "
                   f"({ref['cpu_baseline']['sample']}).\n")
    sl = rd(os.path.join(G, "r2_single_latency.txt"))
    if sl:
        out.append("`tools/single_latency.py`: " + sl.strip().replace("\n", "; ") + ".\n")

    # ---------------- workloads on one GPU
    rows = []
    for f in sorted(glob.glob(os.path.join(G, "r2_multi_*_n1.json"))):
        tag = re.match(r"r2_multi_(.*)_n1\.json", os.path.basename(f)).group(1)
        l = last(f)
        if tag == "static4096" and b:
            l = b  # the headline line above is the one-GPU static4096 row of the final build
        if l:
            rows.append((tag, l))
    if rows:
        out.append("## Workloads on one GPU (`bench.py --workload ...`, five or six batches in flight; `tools/r2_single_sweep.sh`)\n")
        out.append("| workload | shape | solves/s in flight | round 1 | × | ms per step | e2e solves/s | evals / solve | algorithmic % of FP64 peak | exit status (conv / iter / time / nan) |")
        out.append("|---|---|---:|---:|---:|---:|---:|---:|---:|---|")
        for tag, l in rows:
            c = l["config"]
            r1 = R1.get(tag)
            out.append(f"| `{c['workload']}` | N={c['N_hor']}, slots {c['Nstcobs']} static / {c['Ndynobs']} dynamic, active {c['static_per_scene']} + {c['dynamic_per_scene']}, "
                       f"{c['scenes_per_step_per_gpu']} scenes, limits {c['max_inner']}×{c['max_outer']} | {l['value']:,.0f} | {r1:,} | {l['value'] / r1:.2f} | "
                       f"{l['ms_per_step']:.2f} | {l['e2e']['value']:,.0f} | {l['roofline']['evals_per_solve']:.0f} | {100 * l['roofline']['frac']:.1f} | {l['exit_status_hist']} |"
                       if r1 else
                       f"| `{c['workload']}` | N={c['N_hor']} | {l['value']:,.0f} | — | — | {l['ms_per_step']:.2f} | {l['e2e']['value']:,.0f} | {l['roofline']['evals_per_solve']:.0f} | {100 * l['roofline']['frac']:.1f} | {l['exit_status_hist']} |")
        out.append("")
        out.append("All rows are the shipped build except `dynamic8192` (the build one step earlier, `TT_OPT=63`, without the inlined L-BFGS butterflies; "
                   "the GPU budget of the round ended before that 10-second run could be repeated).\n")
        out.append("The sweep shapes of BASELINE `configs[4]` have their own compiled kernels since round 2 (`TTMPC_SOLVE_SHAPES`); "
                   "`dynamic8192` is the per-GPU shard of `configs[2]` with 2000 × 20 iteration limits (an assumption, stated in the bench line's `config.iteration_limits`).\n")

    # ---------------- multi GPU: the lines of ONE 8-GPU box (tools/r2_multi.sh), kept under profiles/
    per_tag = {}
    for l in jl(os.path.join(P, "r2_bench_lines_workloads_and_1_2_4_8_gpus.json")):
        per_tag.setdefault(l["config"]["workload"], {})[l["n_gpus"]] = l
    multi = [(tag, per_n) for tag, per_n in sorted(per_tag.items()) if len(per_n) > 1]
    if multi:
        out.append("## Multi-GPU (weak scaling: every rank solves its own batches, `torch.distributed.run ... bench.py --gpus N`)\n")
        out.append("All rows from ONE 8-GPU box (`tools/r2_multi.sh`, build of commit 2abe7e3, six batches in flight; the single-GPU tables above are "
                   "from the final build of the third session, ≈ 20 % faster on `static4096`: 673 k against 552 k solves/s on one GPU; the 8-GPU budget of the round was spent before it). `profiles/r2_bench_lines_workloads_and_1_2_4_8_gpus.json` holds the lines.\n")
        fin = jl(os.path.join(P, "r2_bench_lines_final_build_1_2_gpus.json"))
        if len(fin) == 2:
            a, c2 = fin
            out.append(f"Final build of the third session, one 2-GPU box (`profiles/r2_bench_lines_final_build_1_2_gpus.json`): {a['value']:,.0f} solves/s on one GPU "
                       f"({a['ms_per_step']:.2f} ms per step), **{c2['value']:,.0f}** on two ({c2['ms_per_step']:.2f} ms, efficiency {c2['value'] / (2 * a['value']):.3f}; "
                       f"e2e {c2['e2e']['value']:,.0f}).\n")
        out.append("| workload | GPUs | solves/s (whole job) | efficiency vs N × one GPU | ms per step (max over ranks) | per-rank ms (min / mean / max) | e2e solves/s |")
        out.append("|---|---:|---:|---:|---:|---|---:|")
        for tag, per_n in multi:
            base = per_n.get(1)
            for n, l in sorted(per_n.items()):
                eff = f"{l['value'] / (n * base['value']):.3f}" if base else "—"
                pr = l.get("per_rank", {}).get("ms_per_step_min_mean_max", [0, 0, 0])
                out.append(f"| `{l['config']['workload']}` | {n} | {l['value']:,.0f} | {eff} | {l['ms_per_step']:.2f} | "
                           f"{pr[0]:.2f} / {pr[1]:.2f} / {pr[2]:.2f} | {l['e2e']['value']:,.0f} |")
        out.append("")
        out.append("No collective in the solve; NCCL carries the barrier, the max-over-ranks time and the gather of per-rank times, counters and "
                   "exit-status histograms. Every rank rotates through the same seeded batches starting at a different one, so the ranks carry equal work "
                   "(round 1 gave every rank its own seeds: 0.88 efficiency at 8 GPUs was the unluckiest rank's tail).\n")

    # ---------------- parity
    for fn, title in (("r2_parity_distribution_gpu.json", "GPU"), ("r2_parity_distribution_cpu.json", "kernel operation order on the CPU (WARP-order oracle, bit-identical to the GPU)")):
        path = os.path.join(P, fn)
        if os.path.exists(path):
            out.append(f"## Solver parity — {title} against the reference operation order, and the reference order's own sensitivity\n")
            out += parity_table(json.load(open(path)))
            out.append("")
            out.append("`tools/parity_report.py`; seeded samples of the BASELINE workloads. Reference order = sequential sums, libm, unfused products like Rust, "
                       "literal two-loop L-BFGS (`oracle/ttmpc_oracle.c`). The second row of each pair is the reference-order oracle against ITSELF with every entry of "
                       "`p` moved by one ulp: the 1e-4 / 1e-6 bars of `north_star` are below that floor, so they are printed, not asserted; the tests assert the "
                       "distribution (`tests/test_parity_distribution.py`, `tests/test_gpu_parity.py::test_gpu_against_reference_order_distribution`). "
                       "Against the WARP-order oracle the GPU is bit-identical on every scene (`tools/stress_parity.py`: 4096 / 4096).\n")
            break

    q = last(os.path.join(G, "r2_qnet.json"))
    if q:
        out.append("## DQN companion\n")
        out.append(f"{q['n_envs']} environments: observation + Q-network {q['ms_observe_plus_qnet_mma']:.2f} ms with the network on the tensor cores "
                   f"(`qnet_mma_kernel`, 15 µs of it) against {q['ms_observe_plus_qnet_fma']:.2f} ms on the FMA pipe; max |ΔQ| between the two {q['max_abs_dq']:.1e}, "
                   f"actions equal on {100 * q['actions_equal']:.1f} %; against torch fp32 on the reference's trained model max |ΔQ| 8.6e-6 (`tools/qnet_diag.py`).\n")
    fl = list({r["robots"]: r for r in jl(os.path.join(G, "r2_fleet.json"))}.values())
    if fl:
        out.append("## Closed loop on the device (`FleetPlanner.step`, `tools/bench_fleet.py`; multipliers persist from step to step like in the reference)\n")
        out.append(f"Each leg drives the same seeded fleet until every robot has stopped or {fl[0]['max_steps']} steps have run. "
                   "Options: 0 = none, W = warm start, S = skip stopped robots. The legs ran interleaved (0 W S WS WS S W 0); "
                   f"each row is the mean of an option's two legs. {fl[0]['gpu']}, power limit {fl[0]['power_limit']}.\n")
        out.append("Robots with contact: robots whose swept clearance was <= 0 in some step (the default monitor of "
                   "`FleetPlanner.enable_monitor`, run outside the timed window; – where the line has no count).\n")
        out.append("| robots | options | steps | drive time (s) | ms / step p50 | p90 | PANOC iterations | reached / failed / running | robots with contact |")
        out.append("|---:|:--|---:|---:|---:|---:|---:|:--|---:|")
        for r in fl:
            for leg, m in r["mean"].items():
                out.append(f"| {r['robots']} | {leg} | {m['steps']} | {m['drive_ms'] / 1e3:.2f} | {m['step_ms_p50']:.1f} | {m['step_ms_p90']:.1f} | "
                           f"{m['panoc_iters']:,.0f} | {m['reached']} / {m['failed']} / {m['running']} | {m.get('contact', '–')} |")
        out.append("")
    out += monitor_section(last(os.path.join(G, "r2_monitor.json")))
    out += missions_section(list({r["robots"]: r for r in jl(os.path.join(G, "r2_missions.json"))}.values()),
                            last(os.path.join(G, "r2_missions_profile.json")))
    hy = last(os.path.join(G, "r2_hybrid.json"))
    if hy:
        out.append("## DQN-boosted closed loop (BASELINE `configs[3]`, `tools/bench_hybrid.py`)\n")
        out.append(f"{hy['envs']} environments: {hy['step_ms_p50']:.1f} ms per control step (p90 {hy['step_ms_p90']:.1f}) = {hy['env_steps_per_s']:,.0f} env-steps/s "
                   f"(round 1: 1,351,483); DQN part (internal observation + lidar + Q-net + hint rollout) {hy.get('dqn_part_ms_p50', 0):.2f} ms of it; "
                   f"{hy.get('mean_inner_iters', 0):.0f} PANOC iterations per solve.\n")
    out += lidar_moving_section(last(os.path.join(G, "r2_lidar_moving.json")), jl(os.path.join(G, "r2_hybrid_lidar.json")),
                                jl(os.path.join(G, "r2_hybrid_drive.json")))
    out += world_section(jl(os.path.join(G, "r2_world.json")))
    open(os.path.join(ROOT, "BENCH.md"), "w").write("\n".join(out) + "\n")
    print("\n".join(out))


if __name__ == "__main__":
    main()
