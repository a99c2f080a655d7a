"""CPU side of the fleet-step options: the warm-start rule of the test oracle on hand-made rows, and
the ctypes mirror of struct ttmpc_fleet against the C header."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from trajtrack_mpcndqn_rlboost_b200 import _lib
from tests.fleet_options_ref import warm_start

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_warm_start_rule_on_hand_made_rows():
    N = 4
    u = np.arange(4 * 2 * N, dtype=np.float64).reshape(4, 2 * N) + 0.5
    status = np.array([0, 0, 1, 2], np.int32)          # RUNNING, RUNNING, REACHED, FAILED
    exit_status = np.array([0, 1, 0, 3], np.int32)     # converged, not converged, ...
    out = warm_start(status, u, exit_status)
    # converged: shifted by one step (v, w pairs), the last control repeated
    assert np.array_equal(out[0], np.concatenate([u[0, 2:], u[0, -2:]]))
    assert np.array_equal(out[0, :2], u[0, 2:4]) and np.array_equal(out[0, -4:-2], out[0, -2:])
    # not converged: zeros
    assert np.array_equal(out[1], np.zeros(2 * N))
    # stopped robots: left alone, whatever their exit status
    assert np.array_equal(out[2:], u[2:])
    assert np.array_equal(u[0], np.arange(2 * N) + 0.5), "the input rows must not change"
    # every exit status but CONVERGED zeroes a running robot's row
    for code in (1, 2, 3):
        assert not warm_start(np.zeros(1, np.int32), u[:1], np.array([code])).any()
    # horizon 1: the shift keeps the only control
    u1 = np.array([[0.25, -0.5]])
    assert np.array_equal(warm_start(np.zeros(1, np.int32), u1, np.zeros(1, np.int32)), u1)


def test_fleet_struct_layout_and_version_match_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "ttmpc.h"\n'
                   'int main(void) { printf("%zu %zu %zu %d %d %d\\n", sizeof(ttmpc_fleet), '
                   'offsetof(ttmpc_fleet, options), offsetof(ttmpc_fleet, action_steps), TTMPC_FLEET_WARM_START, '
                   'TTMPC_FLEET_SKIP_STOPPED, TTMPC_VERSION); return 0; }\n')
    exe = tmp_path / "layout"
    try:
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    except (OSError, subprocess.CalledProcessError) as e:
        pytest.fail(f"could not compile against include/ttmpc.h: {e}")
    size, off_options, off_action, warm, skip, version = map(int, subprocess.check_output([str(exe)]).split())
    assert C.sizeof(_lib.TtmpcFleet) == size
    assert _lib.TtmpcFleet.options.offset == off_options == off_action + 4
    assert (_lib.FLEET_WARM_START, _lib.FLEET_SKIP_STOPPED) == (warm, skip)
    assert version == 102 == _lib.load().ttmpc_version()
    assert _lib.TtmpcFleet().options == 0
