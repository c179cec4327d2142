#!/usr/bin/env python
"""Generate golden vectors by running the REFERENCE'S OWN PYTHON CODE.

Run where the reference's sources are, SAG_REFERENCE naming their directory:

    SAG_REFERENCE=<reference checkout> python tests/golden/make_golden.py

The reference (lasgroup/safe-adaptation-gym) is pure Python on top of dm_control/MuJoCo, gym and
xmltodict, none of which is installable here.  Everything the reference computes itself -- lidar
(safe_adaptation_gym.py:174-223), observation assembly (:120-139), cost (world.py:144-155), every
task's reward / goal logic (tasks/*.py), layout rejection sampling (world.py:172-217,
utils.py:28-70), yaw draw order (world.py:108-137), the step loop (safe_adaptation_gym.py:56-83) and
the benchmark task sampler (benchmark/__init__.py, task_sampler.py) -- is executed UNMODIFIED from
the directory SAG_REFERENCE names.  Only the third-party layer is replaced:

  * ``dm_control`` / ``gym`` / ``xmltodict`` are stub modules;
  * ``MujocoBridge`` (mujoco_bridge.py, the reference's one and only door to the simulator) is
    replaced by ``FakeBridge`` below, which answers the same methods from the oracle's physics
    (oracle/sag_oracle.c: orc_phys_*), and ``Robot`` by constants from point.xml;
  * ``numpy.random.RandomState`` is wrapped so that every draw is recorded; the oracle replays the
    recorded stream (orc_env_set_replay), which pins the ORDER and USE of every random number.

So a golden trajectory = reference Python logic over oracle physics.  tests/test_golden.py then
requires the oracle's own restatement of that logic (orc_env_reset / orc_env_step) to reproduce
obs / reward / cost / layouts to 1e-12.  What this cannot pin is the physics itself (MuJoCo).
"""
import json
import os
import sys
import types
import xml.etree.ElementTree as ET

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("SAG_REFERENCE", "")
sys.path.insert(0, ROOT)

import oracle as O  # noqa: E402

# --------------------------------------------------------------------------------------------
# stub third-party modules
# --------------------------------------------------------------------------------------------


class PhysicsError(RuntimeError):
    pass


def _tolerance(x, bounds=(0.0, 0.0), margin=0.0, sigmoid="gaussian", value_at_margin=0.1):
    # dm_control.utils.rewards.tolerance with margin == 0 [EXT]: 1 inside the bounds, else 0
    assert margin == 0.0
    lower, upper = bounds
    return float(lower <= x <= upper)


class _Elem:
    """Small stand-in for dm_control.mjcf elements: keeps the attributes and children a task adds and serialises
    them, so the rod / ball bodies (roll_rod.py:24-41, dribble_ball.py:21-39) reach FakeBridge.rebuild as XML like
    every other body; haul_box.py:16-29 only builds a tendon whose text is never parsed."""

    def __init__(self, tag="root", **attrs):
        self._tag, self._attrs, self._children = tag, attrs, []

    def __getattr__(self, k):
        if k.startswith("_"):
            raise AttributeError(k)
        child = _Elem(k)
        self._children.append(child)
        return child

    def add(self, tag, **kw):
        child = _Elem(tag, **kw)
        self._children.append(child)
        return child

    @staticmethod
    def _text(v):
        if isinstance(v, str):
            return v
        if isinstance(v, (list, tuple, np.ndarray)):
            return " ".join(repr(float(t)) for t in np.asarray(v, dtype=np.float64).ravel())
        return repr(v)

    def to_xml_string(self):
        attrs = "".join(' %s="%s"' % (k, self._text(v)) for k, v in self._attrs.items())
        inner = "".join(c.to_xml_string() for c in self._children)
        return "<%s%s>%s</%s>" % (self._tag, attrs, inner, self._tag)


def install_stubs():
    if not os.path.isdir(REF):  # otherwise "" would put the working directory on sys.path and the import fail late
        sys.exit("SAG_REFERENCE must name the directory of the reference's sources (safe_adaptation_gym/ inside it); "
                 "got %r" % REF)
    dm = types.ModuleType("dm_control")
    mujoco = types.ModuleType("dm_control.mujoco")
    def _quat2mat(m, q):  # mujoco.mju_quat2Mat [EXT]: row-major 3x3 of a unit quaternion (w, x, y, z)
        w, x, y, z = q
        m[:] = [w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y),
                2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x),
                2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z]
    mujoco.mju_quat2Mat = _quat2mat
    mjcf = types.ModuleType("dm_control.mjcf")
    mjcf.RootElement = _Elem
    rl = types.ModuleType("dm_control.rl")
    control = types.ModuleType("dm_control.rl.control")
    control.PhysicsError = PhysicsError
    utils = types.ModuleType("dm_control.utils")
    rewards = types.ModuleType("dm_control.utils.rewards")
    rewards.tolerance = _tolerance
    dm.mujoco, dm.mjcf, dm.rl, dm.utils = mujoco, mjcf, rl, utils
    rl.control = control
    utils.rewards = rewards
    for name, mod in [("dm_control", dm), ("dm_control.mujoco", mujoco), ("dm_control.mjcf", mjcf),
                      ("dm_control.rl", rl), ("dm_control.rl.control", control), ("dm_control.utils", utils),
                      ("dm_control.utils.rewards", rewards)]:
        sys.modules[name] = mod
    gym = types.ModuleType("gym")
    core = types.ModuleType("gym.core")
    spaces = types.ModuleType("gym.spaces")

    class Env:
        pass

    class Box:
        def __init__(self, low, high, shape=None, dtype=np.float32):
            self.low, self.high, self.shape, self.dtype = low, high, shape, dtype

    gym.Env, core.ActType, core.ObsType, spaces.Box = Env, object, object, Box
    gym.core, gym.spaces = core, spaces
    sys.modules.update({"gym": gym, "gym.core": core, "gym.spaces": spaces})
    sys.modules["xmltodict"] = types.ModuleType("xmltodict")
    sys.path.insert(0, REF)


# --------------------------------------------------------------------------------------------
# recording RandomState
# --------------------------------------------------------------------------------------------
EVENTS = []
_RealRS = np.random.RandomState


class RecRS(_RealRS):
    """numpy RandomState that logs every draw the reference makes (legacy formulas restated so that
    the unit uniform behind each draw is known: uniform = low + (high - low) * random_sample())."""

    def uniform(self, low=0.0, high=1.0, size=None):
        assert size is None
        u = float(self.random_sample())
        EVENTS.append(("uniform", u))
        return low + (high - low) * u

    def normal(self, loc=0.0, scale=1.0, size=None):
        v = _RealRS.normal(self, loc, scale, size)
        EVENTS.append(("normal", [float(x) for x in np.atleast_1d(v)]))
        return v

    def choice(self, a, size=None, replace=True, p=None):
        assert size is None and p is None and isinstance(a, (int, np.integer))
        k = int(_RealRS.choice(self, a))
        EVENTS.append(("choice", int(a), k))
        return k

    def standard_cauchy(self, size=None):
        v = _RealRS.standard_cauchy(self, size)
        EVENTS.append(("cauchy", None))
        return v


def replay_stream(events):
    """Flatten recorded events into the unit-uniform stream the oracle replays."""
    out = []
    for ev in events:
        if ev[0] == "uniform":
            out.append(ev[1])
        elif ev[0] == "normal":
            out.extend(ev[1])  # replayed verbatim as the noise values (orc_env_step)
        elif ev[0] == "choice":
            out.append((ev[2] + 0.5) / ev[1])
        # cauchy: task.ctrl_scale draw (task.py:85-89) -- not consumed by the oracle (scale cfg 0)
    return out


# --------------------------------------------------------------------------------------------
# FakeRobot / FakeBridge: MujocoBridge's interface answered from the oracle physics
# --------------------------------------------------------------------------------------------
class FakeRobot:  # robot.py:8-59 evaluated on point.xml / car.xml
    def __init__(self, path):
        self.base_path = path
        self.name = os.path.splitext(os.path.basename(path))[0]
        assert self.name in ("point", "car")
        self.z_height = 0.1
        self.nu = 2
        self.hinge_pos_names, self.hinge_vel_names, self.ballquat_names, self.ballangvel_names = [], [], [], []
        if self.name == "point":
            self.geom_names = {"robot", "pointarrow"}
            self.nq = self.nv = 3
        else:  # car.xml:16-31 geoms, :37-38 joint sensors
            self.geom_names = {"robot", "back_bumper", "back_connector", "front_bumper", "front_connector", "left", "right", "rear"}
            self.nq, self.nv = 13, 11
            self.ballquat_names, self.ballangvel_names = ["ballquat_rear"], ["ballangvel_rear"]


_ROBOT_GEOMS = {"point": ["robot", "pointarrow"],
                "car": ["robot", "back_bumper", "back_connector", "front_bumper", "front_connector", "left", "right", "rear"]}
_PREFIX_TYPE = [("hazards", O.HAZARD), ("vases", O.VASE), ("gremlins", O.GREMLIN), ("pillars", O.PILLAR),
                ("goal", O.GOAL), ("buttons", O.BUTTON), ("box", O.BOX)]
_SENSOR_SLICE = {"accelerometer": slice(0, 3), "velocimeter": slice(3, 6), "gyro": slice(6, 9),
                 "magnetometer": slice(9, 12), "ballangvel_rear": slice(12, 15)}


class _NamedView(dict):
    """physics.named.model.geom_user / geom_rgba stand-in: assignments are stored as float arrays, as a
    write into the MuJoCo model array would be (press_buttons.py:78-91 assigns Python lists)."""

    def __setitem__(self, k, v):
        dict.__setitem__(self, k, np.atleast_1d(np.asarray(v, dtype=np.float64)))


class _Physics:
    def __init__(self, bridge):
        self.b = bridge

    def step(self, nstep=1):
        self.b.env.phys_step(nstep)
        if self.b.env.error:
            raise PhysicsError("oracle physics error")

    def forward(self):
        self.b.env.forward()


class FakeBridge:
    TASK = "go_to_goal"  # set by the harness before construction (selects tendon / dyn params)

    def __init__(self, robot, addition_render_objects_specs=None, config=None):
        self.robot = robot
        self.env = O.OracleEnv(robot.name, FakeBridge.TASK)
        self.env.clear_world()
        self.physics = _Physics(self)
        self.names, self.z = [], {}
        self.user_groups, self.geom_rgba, self.site_rgba = _NamedView(robot=np.array([0.0])), _NamedView(), _NamedView()
        self.actuator_ctrlrange = np.array([[-1.0, 1.0], [-1.0, 1.0]])
        self.nu = 2
        self.checked_sizes = []

    def rebuild(self, config):  # mujoco_bridge.py:170-175 + _build :41-168
        e = self.env
        e.clear_world()
        self.names, self.z = [], {}
        self.user_groups = _NamedView(robot=np.array([0.0]))
        for name, (body_strs, weld) in config["bodies"].items():
            body = ET.fromstring(body_strs[0])
            if name.startswith("gremlins"):
                # primitive_objects.py:57-86: free body + mocap body + weld.  The mocap BODY has no pos (world origin), its
                # geom carries the offset and does not collide; the weld's solref is what the oracle's weld rows use
                mocap = ET.fromstring(body_strs[1])
                w = ET.fromstring(weld)
                assert mocap.get("mocap") == "true" and mocap.get("pos") is None and mocap.get("name") == name + "mocap"
                mg = mocap.find("geom")
                assert mg.get("contype") == "0" and mg.get("conaffinity") == "0" and mg.get("pos") == body.get("pos")
                assert (w.get("body1"), w.get("body2")) == (name, name + "mocap")
                assert [float(t) for t in w.get("solref").split()] == [0.02, 1.5]
                assert float(body.find("geom").get("density")) == 0.001
            else:
                assert not weld
            if name == "circle":  # unsupervised.py:25-46: visual only, never in the layout
                continue
            pos = [float(t) for t in body.get("pos").split()]
            quat = [float(t) for t in body.get("quat").split()] if body.get("quat") else [1.0, 0.0, 0.0, 0.0]
            yaw = 2.0 * np.arctan2(quat[3], quat[0])  # the rod's euler = "90 0 0" lays the cylinder along y: planar yaw 0
            # the XML carries rot2quat(theta) (utils.py:92-94); recover the exact drawn theta = 2*pi*u from the
            # recorded draws so that the injected world is bit-identical to what the oracle's own reset builds
            cands = [0.0 + (2 * np.pi - 0.0) * ev[1] for ev in EVENTS if ev[0] == "uniform"]
            if cands:
                best = min(cands, key=lambda c: abs(((c - yaw + np.pi) % (2 * np.pi)) - np.pi))
                if abs(((best - yaw + np.pi) % (2 * np.pi)) - np.pi) < 1e-9:
                    yaw = best
            geom = body.find("geom")
            type_ = next(t for p, t in _PREFIX_TYPE if name.startswith(p))
            if type_ == O.BOX:  # roll_rod.py:33 cylinder, dribble_ball.py:29 sphere
                type_ = {"box": O.BOX, "cylinder": O.ROD, "sphere": O.BALL}[geom.get("type")]
            group = int(float(geom.get("user")))
            size = [float(t) for t in geom.get("size").split()]
            self.checked_sizes.append((name, geom.get("type"), size, pos[2]))
            e.add_obj(type_, pos[0], pos[1], yaw, 0.0, group)
            self.names.append(name)
            self.z[name] = pos[2]
            self.user_groups[name] = np.array([float(group)])
        rx, ry = config["robot_xy"]
        e.robot_state = [rx, ry, config["robot_rot"], 0, 0, 0]
        e.robot_ext = [0, 0, 1, 0, 0, 0]
        if config.get("modify_tree"):  # go_to_goal_damping.py / go_to_goal_motor.py
            damp, gear = 0.01, 0.3
            for (ns, id_), (attr, value) in config["modify_tree"]:
                if ns == "joint" and attr == "damping":
                    damp = float(value)
                if ns == "actuator" and attr == "gear":
                    gear = float(str(value).split()[0])
            e.L.orc_env_set_dyn_params(e.h, damp, gear)
        scale = config.get("robot_ctrl_range_scale")
        if scale is not None:
            self.actuator_ctrlrange = np.array([[-1.0, 1.0], [-1.0, 1.0]]) * np.asarray(scale)[:, None]
        self.has_tendon = "tendon" in config.get("others", {})
        e.forward()

    # getters ---------------------------------------------------------------------------------
    def _slot(self, name):
        return self.names.index(name)

    def get_sensor(self, name):
        if name == "ballquat_rear":
            return self.env.robot_ext[2:6]
        return self.env.sensors()[_SENSOR_SLICE[name]]

    def body_pos(self, name):
        if name == "robot":
            s = self.env.robot_state
            return np.array([s[0], s[1], self.robot.z_height])
        o = self.env.get_obj(self._slot(name))
        return np.array([o.x, o.y, self.z[name]])

    def body_mat(self, name):
        assert name == "robot"
        th = self.env.robot_state[2]
        c, s = np.cos(th), np.sin(th)
        return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])

    def _com_offset(self):  # body-frame COM offset of the whole robot (masses from point.xml / car.xml, density rule)
        if self.robot.name == "point":
            return 0.001 * 0.1 / (4.0 / 3.0 * np.pi * 0.1 ** 3 + 0.001), 0.0
        m = np.array([0.02, 0.002, 3e-4, 0.001, 6e-4] + [np.pi * 0.05 ** 2 * 0.05 * 5] * 2 + [4 / 3 * np.pi * 0.05 ** 3 * 5])
        y = np.array([0.0, 0.15, 0.125, -0.165, -0.13, 0.1, 0.1, -0.1])
        x = np.array([0.0, 0.0, 0.0, 0.0, 0.0, -0.13, 0.13, 0.0])
        return float((m * x).sum() / m.sum()), float((m * y).sum() / m.sum())

    def body_com(self, name):  # subtree_com of the robot
        s = self.env.robot_state
        cx, cy = self._com_offset()
        return np.array([s[0] + cx * np.cos(s[2]) - cy * np.sin(s[2]), s[1] + cx * np.sin(s[2]) + cy * np.cos(s[2]), 0.1])

    def body_vel(self, name):  # subtree_linvel
        s = self.env.robot_state
        cx, cy = self._com_offset()
        ox, oy = cx * np.cos(s[2]) - cy * np.sin(s[2]), cx * np.sin(s[2]) + cy * np.cos(s[2])
        return np.array([s[3] - s[5] * oy, s[4] + s[5] * ox, 0.0])

    def robot_pos(self):
        return self.body_pos("robot")

    def robot_mat(self):
        return self.body_mat("robot")

    def robot_vel(self):
        return self.body_vel("robot")

    def set_body_pos(self, name, pos):
        self.env.set_obj(self._slot(name), x=float(pos[0]), y=float(pos[1]))

    def set_mocap_pos(self, name, pos):  # mujoco_bridge.py:232-233; world.py:157-165 writes one value to every gremlin's mocap
        assert name.endswith("mocap") and name[:-5] in self.names and float(pos[2]) == 0.0
        self.env.set_mocap_pos(float(pos[0]), float(pos[1]))

    def set_control(self, action):
        self.env.set_control(action)

    @property
    def time(self):
        return self.env.time

    def _geom_name(self, slot, part):
        if slot == -1:
            return _ROBOT_GEOMS[self.robot.name][part]
        n = self.names[slot]
        return n if part == 0 else "col%d" % part

    @property
    def contacts(self):  # mujoco_bridge.py:251-257
        return [(self._geom_name(c.sa, c.ga), self._geom_name(c.sb, c.gb)) for c in self.env.contacts()]

    def robot_contacts(self, group_geom_names):  # mujoco_bridge.py:177-191, restated verbatim
        part_of_robot = lambda name: name in self.robot.geom_names  # noqa
        in_group = lambda name: any(name.startswith(geom) for geom in group_geom_names)  # noqa
        count = 0
        for geom1, geom2 in self.contacts:
            count += int((part_of_robot(geom1) or part_of_robot(geom2)) and (in_group(geom1) or in_group(geom2)))
        return count

    def sync_groups(self):
        """push geom_user edits made by the tasks (press_buttons.py:78-91, collect.py:34) to the oracle"""
        for slot, name in enumerate(self.names):
            self.env.set_obj(slot, group=int(self.user_groups[name][0]))


# --------------------------------------------------------------------------------------------
# harness
# --------------------------------------------------------------------------------------------
def make_env(task_key, config=None, seed=0, robot="point"):
    import safe_adaptation_gym.safe_adaptation_gym as sag
    from safe_adaptation_gym.benchmark import TASKS

    config = dict(config or {})
    gremlins = int(config.pop("num_gremlins", 0))  # not a World key: Task.obstacles[2] of a user-defined task (task.py:70)
    task_cls = TASKS[task_key]
    if gremlins:
        base_obstacles = list(task_cls().obstacles)
        task_cls = type(task_cls.__name__ + "WithGremlins", (task_cls,),
                        {"obstacles": property(lambda self: [base_obstacles[0], base_obstacles[1], gremlins, base_obstacles[3]])})

    sag.Robot = FakeRobot
    sag.MujocoBridge = FakeBridge
    FakeBridge.TASK = task_key
    np.random.RandomState = RecRS
    try:
        env = sag.SafeAdaptationGym("xmls/%s.xml" % robot, config=config, render_lidars_and_collision=False)
        del EVENTS[:]
        env.seed(seed)
        env.set_task(task_cls())
    finally:
        pass
    return env


def policy(env, rng, mode):
    """drive-to-target controller + noise so that goals, hazards and contacts are actually visited"""
    b = env.mujoco_bridge
    s = b.env.robot_state
    task = env._world.task
    target = None
    name = type(task).__name__
    if hasattr(task, "_goal_button") and getattr(task, "_goal_button", None) is not None and "Collect" not in name:
        target = b.body_pos(task._goal_button)[:2]
    elif "Collect" in name:
        act = sorted(task._active_buttons)
        target = b.body_pos(act[0])[:2] if act else None
    elif "box" in b.names and "Haul" not in name:
        box = b.body_pos("box")[:2]
        goal = b.body_pos("goal")[:2]
        d = goal - box
        target = box - 0.35 * d / (np.linalg.norm(d) + 1e-9)
        if np.linalg.norm(target - s[:2]) < 0.15:
            target = goal
    elif "goal" in b.names:
        target = b.body_pos("goal")[:2]
    if target is None or mode == "random":
        return rng.uniform(-1, 1, 2)
    d = target - s[:2]
    if env.robot.name == "car":  # differential drive; the car's front is body -y (car.xml:19-20)
        err = np.arctan2(d[1], d[0]) - (s[2] - np.pi / 2)
        err = (err + np.pi) % (2 * np.pi) - np.pi
        fwd = np.clip(1.0 - abs(err), 0.0, 1.0) * 0.02
        a = np.array([fwd + 0.01 * np.clip(err, -1, 1), fwd - 0.01 * np.clip(err, -1, 1)])
        return np.clip(a + 0.003 * rng.normal(size=2), -1, 1)
    err = np.arctan2(d[1], d[0]) - s[2]
    err = (err + np.pi) % (2 * np.pi) - np.pi
    a = np.array([np.clip(1.0 - abs(err), 0.02, 1.0), np.clip(2.0 * err, -1, 1)])
    return np.clip(a + 0.2 * rng.normal(size=2), -1, 1)


def record_episode(task_key, seed, steps, mode="drive", config=None, second_reset=True, robot="point"):
    env = make_env(task_key, config=config, seed=seed, robot=robot)
    b = env.mujoco_bridge
    rng = _RealRS(1234 + seed)
    segs = []
    n_seg = 2 if second_reset else 1
    for seg in range(n_seg):
        if seg == 1:
            env.reset()  # safe_adaptation_gym.py:85-107: seed += 1, same task instance
        b.sync_groups()
        obs0 = env.observation
        layout = {"robot": b.env.robot_state.tolist(), "robot_ext": b.env.robot_ext.tolist(), "objects": b.env.objects().tolist(),
                  "task_state": b.env.task_state.tolist()}
        actions, obs, rew, cost, states = [], [], [], [], []
        for t in range(steps):
            a = policy(env, rng, mode)
            o, r, done, info = env.step(a)
            b.sync_groups()
            actions.append(a.tolist())
            obs.append(np.asarray(o, dtype=np.float64).tolist())
            rew.append(np.atleast_1d(np.asarray(r, dtype=np.float64)).tolist())
            cost.append(float(info["cost"]))
            states.append(b.env.robot_state.tolist())
            assert not done
        segs.append({"obs0": np.asarray(obs0).tolist(), "layout": layout, "actions": actions, "obs": obs,
                     "reward": rew, "cost": cost, "robot": states,
                     "final_objects": b.env.objects().tolist()})
    out = {"task": task_key, "robot": robot, "seed": seed, "config": config or {}, "replay": replay_stream(EVENTS),
           "segments": segs, "sizes": [[n, t, s, z] for n, t, s, z in b.checked_sizes[:40]]}
    np.random.RandomState = _RealRS
    return out


def lidar_kats():
    """SafeAdaptationGym._lidar called directly (unbound) on analytic positions."""
    import safe_adaptation_gym.safe_adaptation_gym as sag

    class B:
        def __init__(self, pos, yaw):
            self.p, self.y = pos, yaw

        def robot_pos(self):
            return np.array([self.p[0], self.p[1], 0.1])

        def robot_mat(self):
            c, s = np.cos(self.y), np.sin(self.y)
            return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])

    class S:
        NUM_LIDAR_BINS = 16
        LIDAR_MAX_DIST = 5.0

    rng = _RealRS(7)
    cases = []
    for k in range(200):
        n = int(rng.randint(1, 22))
        rp = rng.uniform(-2, 2, 2)
        yaw = float(rng.uniform(-np.pi, 3 * np.pi))
        pts = rng.uniform(-2.5, 2.5, (n, 2))
        if k % 10 == 0:  # far objects: sensor clamps at 0
            pts[0] = rp + np.array([6.0, 0.3])
        if k % 7 == 0:  # exactly on a bin edge in the ego frame (yaw 0)
            yaw = 0.0
            pts[0] = rp + 1.5 * np.array([np.cos(np.pi / 8 * (k % 16)), np.sin(np.pi / 8 * (k % 16))])
        s = S()
        s.mujoco_bridge = B(rp, yaw)
        try:
            out = sag.SafeAdaptationGym._lidar(s, [np.array([p[0], p[1], 0.3]) for p in pts])
        except IndexError:  # quirk D7 (angle % 2pi == 2pi); the oracle wraps instead
            continue
        cases.append({"robot": [float(rp[0]), float(rp[1]), yaw], "pts": pts.tolist(), "out": out.tolist()})
    return cases


def layout_goldens():
    """World.sample_layout driven directly (world.py:104-106) for every task, many seeds."""
    from safe_adaptation_gym.benchmark import TASKS
    from safe_adaptation_gym.world import World
    from safe_adaptation_gym.utils import ResamplingError

    out = []
    for task_key in sorted(TASKS):
        if task_key in ("roll_rod", "dribble_ball"):
            pass
        for seed in range(6):
            del EVENTS[:]
            rs = RecRS(seed)
            world = World(rs, TASKS[task_key](), FakeRobot("xmls/point.xml"), None)
            try:
                cfg = world.sample_layout()
            except ResamplingError:
                out.append({"task": task_key, "seed": seed, "fail": True, "replay": replay_stream(EVENTS)})
                continue
            layout = {k: [float(v[0]), float(v[1])] for k, v in world._layout.items()}
            yaws = {}
            for name, (body_strs, weld) in cfg["bodies"].items():
                quat = ET.fromstring(body_strs[0]).get("quat")
                if quat is None:  # rod / ball built through the mjcf stub (roll_rod.py:24-41): no yaw draw
                    continue
                q = [float(t) for t in quat.split()]
                yaws[name] = float(2.0 * np.arctan2(q[3], q[0]))
            out.append({"task": task_key, "seed": seed, "fail": False, "replay": replay_stream(EVENTS),
                        "layout": layout, "order": list(world._layout.keys()), "robot_rot": float(cfg["robot_rot"]),
                        "yaws": yaws, "keepouts": {k: float(v[1]) for k, v in world._placements.items()}})
    return out


def sampler_goldens():
    from safe_adaptation_gym import benchmark

    out = {}
    for name in ("multitask", "task_adaptation"):
        b = benchmark.make(name, batch_size=30, seed=666)
        out[name] = {"train": [n for n, _ in b.train_tasks], "test": [n for n, _ in b.test_tasks]}
    out["registry"] = sorted(benchmark.TASKS.keys())
    return out


def gremlin_episodes():
    """World.set_mocaps (world.py:157-165) + primitive_objects.get_gremlin run by the reference for a user-defined task
    with Task.obstacles[2] = 2 (no task of the registry has gremlins)."""
    episodes = []
    for task_key, seed, steps, mode, robot in [("go_to_goal", 31, 300, "drive", "point"), ("press_buttons", 32, 250, "drive", "point"),
                                               ("push_box", 33, 250, "drive", "point"), ("go_to_goal", 34, 200, "drive", "car")]:
        ep = record_episode(task_key, seed, steps, mode, config={"action_noise": 0.01, "num_gremlins": 2}, robot=robot)
        print("gremlins", robot, task_key, "return", sum(r[-1] for s in ep["segments"] for r in s["reward"]),
              "cost", sum(sum(s["cost"]) for s in ep["segments"]), "replay", len(ep["replay"]))
        episodes.append(ep)
    np.savez_compressed(os.path.join(HERE, "episodes_gremlins.npz"), data=np.frombuffer(json.dumps(episodes).encode(), dtype=np.uint8))


def main():
    install_stubs()
    os.makedirs(HERE, exist_ok=True)
    if "gremlins" in sys.argv[1:]:  # only the gremlin episodes (the other fixtures are left as they are)
        gremlin_episodes()
        return
    with open(os.path.join(HERE, "lidar_kat.json"), "w") as f:
        json.dump(lidar_kats(), f)
    with open(os.path.join(HERE, "layouts.json"), "w") as f:
        json.dump(layout_goldens(), f)
    with open(os.path.join(HERE, "sampler.json"), "w") as f:
        json.dump(sampler_goldens(), f, indent=1)
    episodes = []
    plan = [("go_to_goal", 3, 400, "drive"), ("go_to_goal", 4, 300, "random"), ("go_to_goal_scarce", 5, 300, "drive"),
            ("go_to_goal_damping", 6, 200, "drive"), ("go_to_goal_motor", 7, 200, "drive"),
            ("catch_goal", 8, 300, "drive"), ("unsupervised", 9, 250, "drive"),
            ("press_buttons", 10, 400, "drive"), ("press_buttons_scarce", 11, 300, "drive"),
            ("collect", 12, 400, "drive"), ("push_box", 13, 400, "drive"), ("push_box_scarce", 14, 300, "drive"),
            ("haul_box", 15, 300, "drive"), ("roll_rod", 16, 400, "drive"), ("dribble_ball", 17, 400, "drive")]
    plan = [(t, s_, n, m, "point") for t, s_, n, m in plan] + [
        ("go_to_goal", 21, 250, "drive", "car"), ("press_buttons", 22, 250, "drive", "car"), ("push_box", 23, 200, "drive", "car"),
        ("haul_box", 24, 150, "drive", "car"), ("unsupervised", 25, 120, "random", "car"),
        ("roll_rod", 26, 200, "drive", "car"), ("dribble_ball", 27, 200, "drive", "car")]
    for task_key, seed, steps, mode, robot in plan:
        ep = record_episode(task_key, seed, steps, mode, config={"action_noise": 0.01}, robot=robot)
        print(robot, task_key, "return", sum(r[-1] for s in ep["segments"] for r in s["reward"]),
              "cost", sum(sum(s["cost"]) for s in ep["segments"]), "replay", len(ep["replay"]))
        episodes.append(ep)
    np.savez_compressed(os.path.join(HERE, "episodes.npz"), data=np.frombuffer(json.dumps(episodes).encode(), dtype=np.uint8))
    gremlin_episodes()


if __name__ == "__main__":
    main()
