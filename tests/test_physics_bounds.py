"""Model-validity bounds of the restated physics (VERDICT r01 item 8): nothing in the planar soft-contact model may gain
energy without bound.  A body struck by a much heavier robot moving at v leaves, in a perfectly elastic collision, with at
most 2 v plus the speed it had; the robots' own speeds are capped by actuator force against joint damping (point:
0.3 * 0.05 / 0.01 = 1.5 m/s, point.xml:7-8,15-16,36) or by traction-limited wheel torque (car: ~1 m/s measured).  So on
scripted drive-into-everything trajectories: robot speed <= 1.1 x terminal, every movable body <= 2.5 x terminal, and no
state ever turns non-finite.  Checked on the oracle here (CPU) and on the CUDA path in tests/test_gpu_parity.py
(bit-identical, so the same trajectories).

Known violation, kept visible instead of hidden: car x dribble_ball.  The ball's solref (0.018, 0.2) (dribble_ball.py:31) is
under-damped, and at the car's 8 ms timestep h * omega_n = 2.3 > 2, outside the stability region of semi-implicit Euler:
a hard hit returns more energy than it took (measured 5.6 m/s against a 1 m/s car).  MuJoCo's own `refsafe` guard only
lifts the time constant to 2 h and would not catch it either; whether real MuJoCo shows the same gain is exactly what
tools/mujoco_crosscheck.py is for.  The point robot (4 ms) is inside the region.
"""
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from common import drive_action

TERMINAL = {"point": 1.5, "car": 1.0}


def _trajectory_bounds(robot, task, seeds=4, steps=400):
    vr = vo = 0.0
    for seed in range(seeds):
        o = O.OracleEnv(robot, task, config={"action_noise": 0.0}, seed=seed, env_gid=0)
        assert o.reset(0) == 0
        rng = np.random.RandomState(seed)
        for t in range(steps):
            obs, rew, cost, done, rc = o.step(drive_action(o, rng))
            assert rc == 0 and not done, (robot, task, seed, t)
            s, ob = o.robot_state, o.objects()
            assert np.isfinite(s).all() and np.isfinite(ob).all() and np.isfinite(obs).all()
            vr = max(vr, float(np.hypot(s[3], s[4])))
            vo = max(vo, float(np.hypot(ob[:, 5], ob[:, 6]).max()))
    return vr, vo


CASES = [(r, t) for r in ("point", "car") for t in ("go_to_goal", "press_buttons", "push_box", "haul_box", "roll_rod", "dribble_ball")]


@pytest.mark.parametrize("robot,task", CASES)
def test_speeds_stay_within_the_elastic_collision_bound(robot, task):
    if (robot, task) == ("car", "dribble_ball"):
        pytest.xfail("under-damped ball solref at the car's 8 ms timestep: see the module docstring / DESIGN.md 4")
    vr, vo = _trajectory_bounds(robot, task)
    assert vr <= 1.1 * TERMINAL[robot], (vr, "robot faster than its actuators allow")
    assert vo <= 2.5 * TERMINAL[robot], (vo, "a struck body left faster than an elastic collision allows")


def test_car_dribble_ball_energy_gain_is_bounded_and_documented():
    """the known violation stays a bounded one: the ball does not exceed 10 m/s and nothing turns non-finite"""
    vr, vo = _trajectory_bounds("car", "dribble_ball")
    assert vr <= 1.1 * TERMINAL["car"] and vo <= 10.0, (vr, vo)


CROSSCHECK = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "mujoco_crosscheck.py")


def test_mujoco_crosscheck_harness_selftest():
    """tools/mujoco_crosscheck.py end to end without MuJoCo: the unmodified reference logic over the oracle's physics against
    the mirrored oracle must agree exactly.  Runs the reference's Python sources: SAG_REFERENCE names their directory."""
    if not os.path.isdir(os.environ.get("SAG_REFERENCE", "")):
        pytest.skip("needs the reference's Python sources (SAG_REFERENCE=<directory>)")
    r = subprocess.run([sys.executable, CROSSCHECK, "--selftest", "--steps", "120", "--seeds", "1"], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count(" OK") == 8   # {point, car} x {free, static, movable, gremlin}


def test_mujoco_crosscheck_reports_not_run_without_mujoco():
    """without the MuJoCo stack the tool reports 'not run' (exit code 3) instead of a result"""
    if all(importlib.util.find_spec(m) for m in ("dm_control", "gym", "xmltodict")):
        pytest.skip("the MuJoCo stack is installed")
    r = subprocess.run([sys.executable, CROSSCHECK], capture_output=True, text=True, timeout=120)
    assert r.returncode == 3 and "NOT RUN" in r.stdout
