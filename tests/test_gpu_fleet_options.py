"""The fleet-step options on the GPU (FleetPlanner.step(warm_start=..., skip_stopped=...), i.e.
TTMPC_FLEET_WARM_START / TTMPC_FLEET_SKIP_STOPPED of ttmpc_fleet_step_device) against the
WARP-order oracle, bit for bit."""
import ctypes as C

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib
from trajtrack_mpcndqn_rlboost_b200.fleet import work_mode
from tests import oracle_lib as O
from tests.fleet_options_ref import OracleFleet

pytestmark = pytest.mark.gpu

SOLVER = dict(max_inner_iterations=40, max_outer_iterations=3)  # some solves end NotConvergedIterations
ARRIVE_AT = 3      # before this step, robots 0-3 are put next to their goals at rest: they stop there


def _make(n, seed, **solver):
    mc = t.Configurator()
    fl = t.scenes.make_fleet(n, seed=seed)
    fp = t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], mode="work", **solver)
    fp.update_static_constraints(fl["static_polys"], per_robot=True)
    fp.set_moving_obstacles(fl["moving_pos"], fl["moving_disp"])
    tuning, base = work_mode(mc, "work")
    fh = O.FleetHost(fp.cfg, fl["init"], fl["goal"], fp.ref_traj.cpu().numpy(), fp.ref_len.cpu().numpy(),
                     fp.stc.cpu().numpy(), tuning, base, mc.low_speed, dyn_cur=fl["moving_pos"], dyn_disp=fl["moving_disp"])
    return fp, OracleFleet(fh, fp.cfg)


def _arrive(fp=None, of=None):
    if fp is not None:
        fp.state[:4, :2] = fp.goal[:4, :2] + 0.01; fp.last_u[:4] = 0.0
    if of is not None:
        of.fh.state[:4, :2] = of.fh.goal[:4, :2] + 0.01; of.fh.last_u[:4] = 0.0


def _device_rows(fp):
    return dict(u=fp.u.cpu().numpy(), y=fp.y.cpu().numpy(), cost=fp.cost.cpu().numpy(),
                exit_status=fp.exit_status.cpu().numpy(), inner=fp.inner.cpu().numpy(),
                pred=fp.pred_states.cpu().numpy())


def _assert_step_equal(fp, of, k):
    fh = of.fh
    assert np.array_equal(fp.p.cpu().numpy(), of.p), f"packed parameters differ at step {k}"
    dev = _device_rows(fp)
    for name, ref in of.res.items():
        assert np.array_equal(dev[name], ref), f"{name} differs at step {k}"
    assert np.array_equal(fp.state.cpu().numpy(), fh.state), f"states differ at step {k}"
    assert np.array_equal(fp.last_u.cpu().numpy(), fh.last_u)
    assert np.array_equal(fp.idx_ref.cpu().numpy(), fh.idx_ref)
    assert np.array_equal(fp.status.cpu().numpy(), fh.status)
    assert np.array_equal(fp.dyn_cur.cpu().numpy(), fh.dyn_cur)
    return dev


def test_warm_start_closed_loop_bit_exact():
    n, steps = 32, 8
    fp, of = _make(n, seed=9, **SOLVER)
    _, cold = _make(n, seed=9, **SOLVER)
    shifted = zeroed = 0
    differs_from_cold = False
    for k in range(steps):
        if k == ARRIVE_AT:
            _arrive(fp, of); _arrive(of=cold)
        prev_exit = of.res["exit_status"].copy()
        fp.step(warm_start=True); fp.torch.cuda.synchronize()
        of.step(warm=True)
        cold.step()
        run = of.fh.status == 0
        if k > 0:   # the guard: shift after a converged solve, zeros after any other
            shifted += int((prev_exit[run] == 0).sum()); zeroed += int((prev_exit[run] != 0).sum())
        _assert_step_equal(fp, of, k)
        if k == 0:
            for name in OracleFleet.FIELDS:
                assert np.array_equal(of.res[name], cold.res[name]), f"warm step 1 differs from the cold one in {name}"
        elif not np.array_equal(of.res["u"][run], cold.res["u"][run]):
            differs_from_cold = True
    assert shifted > 0 and zeroed > 0, (shifted, zeroed)
    assert differs_from_cold
    assert (of.fh.status[:4] == 1).all() and (of.fh.status[4:] == 0).sum() > 0


@pytest.mark.parametrize("warm", [False, True], ids=["skip", "warm+skip"])
def test_skip_stopped_closed_loop_bit_exact(warm):
    n, steps = 32, 8
    fp, of = _make(n, seed=9, **SOLVER)
    prev = None
    stopped_during_loop = 0
    for k in range(steps):
        if k == ARRIVE_AT:
            _arrive(fp, of)
        was_running = fp.status.cpu().numpy() == 0
        fp.step(warm_start=warm, skip_stopped=True); fp.torch.cuda.synchronize()
        of.step(warm=warm, skip=True)   # the oracle solves only the robots RUNNING after the goal test
        dev = _assert_step_equal(fp, of, k)
        skipped = np.setdiff1d(np.arange(n), of.solved)
        stopped_during_loop += int((was_running[skipped]).sum())
        if prev is not None:            # rows of skipped robots hold what the last solve wrote
            for name in OracleFleet.FIELDS:
                assert np.array_equal(dev[name][skipped], prev[name][skipped]), f"{name} of a stopped robot changed at step {k}"
        prev = dev
    assert stopped_during_loop >= 1


def _full_result(n, N, sentinel):
    import torch
    f64 = dict(dtype=torch.float64, device="cuda")
    i32 = dict(dtype=torch.int32, device="cuda")
    bufs = dict(u=torch.full((n, 2 * N), sentinel, **f64), cost=torch.full((n,), sentinel, **f64),
                exit_status=torch.full((n,), -7, **i32), outer=torch.full((n,), -7, **i32),
                inner=torch.full((n,), -7, **i32), fpr=torch.full((n,), sentinel, **f64),
                f1=torch.full((n,), sentinel, **f64), f2=torch.full((n,), sentinel, **f64),
                pen=torch.full((n,), sentinel, **f64), y=torch.full((n, 2 * N), sentinel, **f64),
                pred=torch.full((n, N, 3), sentinel, **f64),
                evals=torch.full((n, 4), -7, dtype=torch.int64, device="cuda"))
    r = _lib.TtmpcResult(u=bufs["u"].data_ptr(), cost=bufs["cost"].data_ptr(), exit_status=bufs["exit_status"].data_ptr(),
                         outer_iters=bufs["outer"].data_ptr(), inner_iters=bufs["inner"].data_ptr(),
                         last_fpr=bufs["fpr"].data_ptr(), f1_infeas=bufs["f1"].data_ptr(), f2_norm=bufs["f2"].data_ptr(),
                         penalty=bufs["pen"].data_ptr(), y=bufs["y"].data_ptr(), pred_states=bufs["pred"].data_ptr(),
                         evals=bufs["evals"].data_ptr())
    return bufs, r


@pytest.mark.parametrize("n,code", [(2048, None), (96, "unrolled"), (96, "small")])
def test_skip_stopped_one_solve_leaves_skipped_rows_untouched(n, code, monkeypatch):
    """One skip-stopped step with every second robot REACHED.  2048 robots exceed the resident warps:
    the rolled build with the dispatch order and the early helpers; 96 robots run on each build."""
    import torch
    if code:
        monkeypatch.setenv("TTMPC_CODE", code)
    fp, of = _make(n, seed=12)
    fp.status[1::2] = 1
    of.fh.status[1::2] = 1
    N = fp.N
    bufs, r = _full_result(n, N, -7.25)
    f = fp._fleet_struct()
    f.options = _lib.FLEET_SKIP_STOPPED
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(fp.lib.ttmpc_fleet_step_device(C.byref(fp.cfg), C.byref(f), fp.p.data_ptr(), 0, C.byref(r), st), "fleet step")
    torch.cuda.synchronize()
    p = O.fleet_pack(of.fh, use_libm=False)
    assert np.array_equal(fp.p.cpu().numpy(), p)
    run = np.flatnonzero(of.fh.status == 0)
    skip = np.flatnonzero(of.fh.status != 0)
    assert len(run) == n // 2
    ref = O.solve_batch(fp.cfg, p[run], threads=8, warp=True)
    pairs = dict(u="u", cost="cost", exit_status="exit_status", outer="outer", inner="inner", fpr="fpr",
                 f1="f1", f2="f2", pen="pen", y="y", pred="pred")
    for dev_name, ref_name in pairs.items():
        d = bufs[dev_name].cpu().numpy()
        assert np.array_equal(d[run], ref[ref_name]), f"{dev_name} of a solved robot differs from the oracle"
        assert (d[skip] == (-7 if d.dtype.kind == "i" else -7.25)).all(), f"{dev_name} of a skipped robot was written"
    ev = bufs["evals"].cpu().numpy()   # clock readings and (with helpers) speculative counts: written or not
    assert (ev[run] != -7).all() and (ev[skip] == -7).all()
    O.fleet_advance(of.fh, bufs["u"].cpu().numpy(), bufs["exit_status"].cpu().numpy(), use_libm=False)
    assert np.array_equal(fp.state.cpu().numpy(), of.fh.state)


def test_unknown_option_bits_are_rejected():
    import torch
    fp, _ = _make(4, seed=3)
    r = fp._result_struct()
    st = torch.cuda.current_stream().cuda_stream
    for bad in (4, 1 << 30, -1):
        f = fp._fleet_struct()
        f.options = bad
        rc = fp.lib.ttmpc_fleet_step_device(C.byref(fp.cfg), C.byref(f), fp.p.data_ptr(), 1, C.byref(r), st)
        assert rc == -2, (bad, rc)  # TTMPC_ERR_BAD_ARG
    torch.cuda.synchronize()
    assert (fp.status.cpu().numpy() == 0).all() and fp.steps == 0
