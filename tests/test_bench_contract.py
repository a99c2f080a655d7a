"""bench.py contract checks that need no GPU: the reference (CPU) arm prints one JSON line with the
keys the driver reads, and the product arm refuses to run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True,
                          text=True, timeout=600, env=e, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = run_bench("--impl", "reference", "--steps", "2", "--warmup", "1", "--cpu-sample", "48")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["unit"] == "solves/s" and line["higher_is_better"] is True
    assert line["metric"] == "batched NMPC solves/sec" and line["config"]["workload"] == "static4096"
    assert line["steps"] == 2 and line["warmup"] == 1 and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "solves/s", "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    assert line["ms_per_step"] > 0 and abs(48 / (line["ms_per_step"] * 1e-3) - line["value"]) < 1e-6 * line["value"]


def test_reference_arm_other_ranks_do_no_work():
    r = run_bench("--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-sample", "8", env={"RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_has_no_cpu_path():
    # the GPU is hidden from the child process, so this holds on a machine with a GPU as well
    r = run_bench("--steps", "1", "--warmup", "1", env={"CUDA_VISIBLE_DEVICES": ""})
    assert r.returncode != 0
    assert "no CPU path" in (r.stderr + r.stdout)


def test_workload_parsing_and_common_config():
    """`--workload` names a BASELINE workload or a configs[4] sweep shape; both arms print the SAME
    `config` object (the driver compares them)."""
    sys.path.insert(0, ROOT)
    import argparse
    import bench
    mc, cfg, w = bench.parse_workload("sweep:N=32,Nstc=10,Ndyn=15")
    assert (cfg.N_hor, cfg.Nstcobs, cfg.Ndynobs, w["n"], w["n_static"], w["n_dynamic"]) == (32, 10, 15, 4096, 4, 3)
    mc, cfg, w = bench.parse_workload("dynamic8192")
    assert (cfg.max_inner_iterations, cfg.max_outer_iterations, w["n"]) == (2000, 20, 8192)
    a = argparse.Namespace(workload="dynamic8192", batches=2)
    c1, c2 = bench.common_config(a, cfg, w, 8192), bench.common_config(a, cfg, w, 64)
    assert c1 == c2 and "ASSUMPTION" in c1["iteration_limits"]          # the long limits are an assumption, said so
    # every rank draws the same seeded batches (equal work); the batch index alone selects the seed
    _, p0, _ = bench.build_workload("static4096", 0, 8, 1)
    _, p5, _ = bench.build_workload("static4096", 5, 8, 1)
    _, q0, _ = bench.build_workload("static4096", 0, 8, 2)
    import numpy as np
    assert np.array_equal(p0, p5) and not np.array_equal(p0, q0)


def test_dump_outputs_writes_float64_and_samples_large_batches(tmp_path):
    """--dump-outputs: every result field as <name>.npy in float64, rows in batch order; a batch over
    the 64 MB cap becomes the same seeded sample of scenes every time."""
    sys.path.insert(0, ROOT)
    import bench
    import numpy as np
    import torch

    def bufs(n, N=20):
        g = torch.Generator().manual_seed(n)
        f = lambda *s: torch.rand(*s, generator=g, dtype=torch.float64)
        i = lambda *s: torch.randint(0, 4, s, generator=g, dtype=torch.int32)
        return dict(u=f(n, 2 * N), y=f(n, 2 * N), cost=f(n), exit_status=i(n), outer=i(n), inner=i(n),
                    fpr=f(n), f1=f(n), f2=f(n), pen=f(n), pred=f(n, N, 3),
                    evals=torch.zeros(n, 4, dtype=torch.int64))

    small = bufs(64)
    bench.dump_outputs(small, str(tmp_path / "small"))
    names = sorted(p.stem for p in (tmp_path / "small").iterdir())
    assert names == sorted(list(bench.DUMP_FIELDS) + ["scene_index"])
    for k in bench.DUMP_FIELDS:
        a = np.load(tmp_path / "small" / f"{k}.npy")
        assert a.dtype == np.float64 and np.array_equal(a, small[k].double().numpy())
    assert np.array_equal(np.load(tmp_path / "small" / "scene_index.npy"), np.arange(64))

    big = bufs(70000)   # ~1.2 kB of results per scene: more than 64 MB in all
    for d in ("a", "b"):
        bench.dump_outputs(big, str(tmp_path / d))
    total = sum(p.stat().st_size for p in (tmp_path / "a").iterdir())
    assert total <= bench.DUMP_LIMIT_BYTES + 256 * len(names)   # + the .npy headers
    idx = np.load(tmp_path / "a" / "scene_index.npy").astype(np.int64)
    assert 0 < len(idx) < 70000 and np.all(np.diff(idx) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "u.npy"), big["u"].numpy()[idx])
    for k in list(bench.DUMP_FIELDS) + ["scene_index"]:
        assert np.array_equal(np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy"))


def test_default_depth_divides_the_step_count():
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert "args.steps % d == 0" in src
    for steps, want in ((20, 5), (24, 6), (12, 6), (16, 8), (7, 7), (11, 6)):
        cand = [d for d in (6, 5, 7, 8, 4) if steps % d == 0]
        assert (cand[0] if cand else 6) == want
