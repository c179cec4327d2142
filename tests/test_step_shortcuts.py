"""The step's contact shortcuts against the oracle, at their edges.

The step kernels skip contact work based on state cached by the previous step (or by the refresh that follows a field
write): the clearance (task_f64 row 7) and the moving mask (task_i32 row 9) select the quiet path (no contact test),
the near path (exact overlap pre-tests on the slots within reach) or the contact path, and the contact passes add a
broad phase.  The oracle runs the full contact pipeline in every substep.  Each case here puts bodies where those
decisions change and requires bit-exact agreement of robot, objects, reward, cost, done and observation every step:
  (a) states injected with set_field, load_state_dict or sag_write_field and stepped at once (no env.observation in
      between), and the write-back of an unchanged state, which must change nothing;
  (b) the quiet / near threshold: for extreme robot states and each collidable kind, the largest initial gap at which
      the oracle lists a contact during the step is found by bisection on the oracle alone, and kernel and oracle step
      from just inside and just outside it;
  (c) the object-pair broad phase: a pushed task body reaching a resting vase or pillar at the bisected gap;
  (d) HaulBox: the tendon becoming taut at the bisected slack.
A shortcut bound that is not conservative makes the kernel skip a contact the oracle lists, and the comparison fails,
however travel_bound, the robot reach or kind_bound are written."""
import numpy as np
import pytest
import torch

import oracle as O
from common import env_state, make_env, make_oracles, oracle_state

PHI = 0.3   # world direction of the centre line from the robot to the body
# farthest footprint point of the robot: (distance from the centre, angle in the body frame)
ROBOT_FAR = {"point": (np.hypot(0.15, 0.05), np.arctan2(0.05, 0.15)),     # arrow corner (point.xml:19)
             "car": (np.hypot(0.155, 0.15), np.arctan2(0.15, 0.155))}     # rear wheel corner (car.xml:23-27)
KIND_TASK = {O.VASE: "go_to_goal", O.PILLAR: "go_to_goal", O.BUTTON: "press_buttons", O.BOX: "push_box",
             O.ROD: "roll_rod", O.BALL: "dribble_ball"}
COLLIDABLE = (O.VASE, O.GREMLIN, O.PILLAR, O.BUTTON, O.BOX, O.ROD, O.BALL)
DELTAS = (1e-9, 1e-6, 1e-3)
SEED = 91


def body_far(kind, cfg):
    """farthest footprint point of a body: (distance from its centre, angle in its frame)"""
    return {O.VASE: (np.sqrt(2.0) * cfg.vases_size, np.pi / 4), O.PILLAR: (cfg.pillars_size, 0.0), O.BUTTON: (0.1, 0.0),
            O.BOX: (1.5 * np.sqrt(2.0) * 0.2, np.pi / 4), O.ROD: (np.hypot(0.08, 0.3), np.arctan2(0.3, 0.08)),
            O.BALL: (0.14, 0.0)}[kind]


def _rot(v, yaw):
    c, s = np.cos(yaw), np.sin(yaw)
    return v[0] * c - v[1] * s, v[0] * s + v[1] * c


def _snapshot(o):
    return o.robot_state, o.robot_ext, o.objects()


def _restore(o, snap):
    rs, ext, objs = snap
    o.robot_state = rs
    o.robot_ext = ext
    for s, row in enumerate(objs):
        o.set_obj(s, x=row[2], y=row[3], yaw=row[4], vx=row[5], vy=row[6], w=row[7])


def _clear_others(o, keep, origin):
    """every collidable body except the slots in `keep` far away from `origin`"""
    for k, (s, t) in enumerate(enumerate(o.slot_types())):
        if t in COLLIDABLE and s not in keep:
            o.set_obj(s, x=origin[0] - 6.0 - 0.7 * k, y=origin[1] - 6.0, vx=0.0, vy=0.0, w=0.0)


def face(robot, kind, cfg, vb=(0.0, 0.0), w=0.0, ext=None, body_v=(0.0, 0.0, 0.0), slot_of=0):
    """Scene: the robot's and the body's farthest footprint points face each other on the centre line; `gap` is the
    distance between those two points.  vb: robot velocity in its body frame, w: yaw rate, body_v: the body's velocity
    (along the centre line, across it, spin).  Every other collidable body is moved away."""
    rf, ra = ROBOT_FAR[robot]
    bf, ba = body_far(kind, cfg)

    def scene(o, gap):
        rs = o.robot_state
        yaw = PHI - ra
        rs[2] = yaw
        rs[3], rs[4] = _rot(vb, yaw)
        rs[5] = w
        o.robot_state = rs
        if ext is not None:
            o.robot_ext = ext
        slot = [s for s, t in enumerate(o.slot_types()) if t == kind][slot_of]
        d = rf + bf + gap
        bvx, bvy = _rot(body_v[:2], PHI)
        o.set_obj(slot, x=rs[0] + d * np.cos(PHI), y=rs[1] + d * np.sin(PHI), yaw=PHI + np.pi - ba, vx=bvx, vy=bvy, w=body_v[2])
        _clear_others(o, {slot}, rs[:2])
    return scene


def teleport(robot, cfg):
    """Scene: the robot moved next to the vase slot that is farthest from every other collidable body; the objects
    are not touched (only the robot field is written)"""
    rf, ra = ROBOT_FAR[robot]
    bf, ba = body_far(O.VASE, cfg)

    def scene(o, gap):
        objs = o.objects()
        col = [s for s in range(len(objs)) if int(objs[s, 0]) in COLLIDABLE]
        iso = lambda s: min(np.hypot(*(objs[s, 2:4] - objs[t, 2:4])) for t in col if t != s)   # noqa: E731
        slot = max((s for s in col if int(objs[s, 0]) == O.VASE), key=iso)
        rs = o.robot_state
        d = rf + bf + gap
        rs[0], rs[1] = objs[slot, 2] - d * np.cos(PHI), objs[slot, 3] - d * np.sin(PHI)
        rs[2] = PHI - ra
        o.robot_state = rs
    return scene


def _lists_contact(o, action, nsub, steps=1, pair=None, moved=None):
    """Does the oracle list a contact during `steps` env steps from its current state: substep by substep
    (physics.step) plus the final forward() of each step.  pair: only a contact between these two object slots
    counts; moved: instead of a contact, this object slot leaves rest (the HaulBox tendon pulling the box)."""
    for _ in range(steps):
        o.set_control(np.clip(np.asarray(action, dtype=np.float64), -1.0, 1.0))
        for k in range(nsub + 1):
            if k < nsub:
                o.phys_step(1)
            else:
                o.forward()
            if moved is not None:
                ob = o.get_obj(moved)
                if ob.vx != 0.0 or ob.vy != 0.0 or ob.w != 0.0:
                    return True
            elif pair is not None:
                if any({c.sa, c.sb} == set(pair) for c in o.contacts()):
                    return True
            elif o.contacts():
                return True
    return False


def bisect_gap(make_oracle, scene, action, nsub, lo=-0.05, hi=0.6, **kw):
    """g*: the largest gap at which the oracle lists a contact (kw: see _lists_contact), to the last bit of the bisection
    bracket.  action=None: the static test (forward() at the injected state)."""
    o = make_oracle()
    snap = _snapshot(o)

    def hit(g):
        _restore(o, snap)
        scene(o, g)
        if action is None:
            o.forward()
            return bool(o.contacts())
        return _lists_contact(o, action, nsub, **kw)
    assert hit(lo) and not hit(hi), (lo, hi)
    while True:
        mid = 0.5 * (lo + hi)
        if mid <= lo or mid >= hi:
            return lo
        if hit(mid):
            lo = mid
        else:
            hi = mid


def nsub_of(robot):
    """substeps per env step, from the oracle: the time one step advances over the time one physics substep does"""
    a, b = O.OracleEnv(robot, "go_to_goal"), O.OracleEnv(robot, "go_to_goal")
    a.reset(0); b.reset(0)
    t0 = a.time
    a.phys_step(1)
    b.step(np.zeros(2))
    return int(round((b.time - t0) / (a.time - t0)))


def terminal_state(robot, task, action, steps=300):
    """The robot's state after `steps` steps of a constant action from rest in an empty world (oracle): body-frame
    velocity, yaw rate and the car's wheel rates / castor quaternion"""
    o = O.OracleEnv(robot, task, config={"action_noise": 0.0})
    o.reset(0)
    for s, t in enumerate(o.slot_types()):
        o.set_obj(s, x=1000.0 + s, y=1000.0)
    rs = o.robot_state
    rs[2:] = 0.0
    o.robot_state = rs
    for _ in range(steps):
        o.step(np.asarray(action, dtype=np.float64))
    rs = o.robot_state
    return _rot(rs[3:5], -rs[2]), rs[5], o.robot_ext


# ------------------------------------------------------------------------------------------------------------------
# the batch side: inject the oracles' states, step both, compare every step
# ------------------------------------------------------------------------------------------------------------------
def write_fields(env, fields, route):
    """fields: {name: tensor}, written in order.  route 'set_field' (env.set_field), 'abi' (sag_write_field on the
    handle, as a C binding does)"""
    for name, value in fields.items():
        if route == "abi":
            fid, dt, lead = env._FIELDS[name]
            t = torch.as_tensor(value).to(device=env.device, dtype=dt).contiguous()
            env._lib.check(env._lib.L.sag_write_field(env._h, fid, env._p(t), env._stream()))
            if env.device.type == "cuda":
                torch.cuda.current_stream(env.device).synchronize()
        else:
            env.set_field(name, value)


def fields_from_oracles(env, orc, names=("objects", "robot")):
    """the batch's fields with every environment's robot / objects replaced by its oracle's"""
    n = env.num_envs
    out = {}
    for name in names:
        f = env.get_field(name).cpu()
        for e, o in enumerate(orc):
            if name == "objects":
                objs = o.objects()
                f[:, :len(objs), e] = torch.from_numpy(objs[:, 2:8].T.copy())
            elif name == "robot":
                f[:, e] = torch.from_numpy(o.robot_state)
            elif name == "robot_ext":
                f[:, e] = torch.from_numpy(o.robot_ext)
        assert f.shape[-1] >= n
        out[name] = f
    return out


def step_both(env, orc, acts, steps, route="set_field", tag=""):
    """`steps` steps of the fixed actions acts [n, 2] on both sides; bit-exact agreement every step"""
    n = env.num_envs
    a_t = torch.from_numpy(acts.astype(np.float32)).to(env.device)
    contacts = 0
    for t in range(steps):
        if route == "abi":
            L = env._lib
            L.check(L.L.sag_step(env._h, env._p(a_t), env._p(env._obs), env._p(env._reward), None, env._p(env._cost),
                                 env._p(env._done), env._stream()))
            obs, rew, cost, done = env._obs, env._reward, env._cost, env._done
        else:
            obs, rew, done, info = env.step(a_t)
            cost = info["cost"]
        obs, rew, cost, done = obs.cpu().numpy(), rew.cpu().numpy(), cost.cpu().numpy(), done.cpu().numpy()
        for e in range(n):
            oobs, orew, ocost, odone, rc = orc[e].step(acts[e].astype(np.float32).astype(np.float64))
            msg = f"{tag} env {e} step {t}"
            assert rc == 0, msg
            assert float(cost[e]) == ocost and bool(done[e]) == odone, msg
            assert float(np.atleast_1d(rew[e])[0]) == orew[0], msg
            np.testing.assert_array_equal(obs[e], oobs.astype(np.float32), err_msg=msg)
            contacts += len(orc[e].contacts())
        r1, o1 = env_state(env)
        ro, oo = oracle_state(orc)
        np.testing.assert_array_equal(r1, ro, err_msg=f"{tag} robot state step {t}")
        np.testing.assert_array_equal(o1, oo, err_msg=f"{tag} object state step {t}")
    return contacts


class Batch:
    """A batch env and its oracles, one (task, scene, gap) per environment"""

    def __init__(self, backend, robot, tasks, config=None):
        self.cfg = dict(config or {})
        self.cfg.setdefault("action_noise", 0.0)
        self.robot, self.tasks = robot, list(tasks)
        self.env = make_env(backend, len(tasks), self.tasks, SEED, self.cfg, robot=robot)
        self.orc = make_oracles(len(tasks), self.tasks, SEED, self.cfg, robot=robot)
        r0, o0 = env_state(self.env)
        ro, oo = oracle_state(self.orc)
        np.testing.assert_array_equal(r0, ro)
        np.testing.assert_array_equal(o0, oo)

    def fresh_oracle(self, e):
        def make():
            o = O.OracleEnv(self.robot, self.tasks[e], config=self.cfg, seed=SEED, env_gid=e)
            assert o.reset(0) == 0
            return o
        return make


# ------------------------------------------------------------------------------------------------------------------
# (a) injected states, stepped without env.observation
# ------------------------------------------------------------------------------------------------------------------
def _injection_cases(robot):
    """(task, scene, gap rule, write robot only, derived-row edit) per environment"""
    cases = []
    for kind in KIND_TASK:   # every collidable kind a registry task holds, overlapping the robot by 1 mm
        cases.append((KIND_TASK[kind], ("face", kind, (0.0, 0.0, 0.0)), "overlap", False, None))
    cases.append(("go_to_goal", ("teleport",), "overlap", True, None))
    for kind in (O.VASE, O.BOX, O.ROD, O.BALL):   # a velocity on a resting body, far from the robot and next to it
        cases.append((KIND_TASK[kind], ("keep", kind, (0.3, 0.1, 0.5)), None, False, None))
        cases.append((KIND_TASK[kind], ("face", kind, (-0.3, 0.0, 0.0)), 0.02, False, None))
    cases.append(("go_to_goal", ("face", O.VASE, (0.0, 0.0, 0.0)), "overlap", False, "clear"))   # clearance +1e30
    cases.append(("push_box", ("keep", O.BOX, (0.3, 0.0, 0.0)), None, False, "movmask"))          # moving mask 0
    return cases


def run_injection(backend, robot, route, steps=4):
    cases = _injection_cases(robot)
    B = Batch(backend, robot, [c[0] for c in cases])
    env, orc, cfg = B.env, B.orc, O.default_config(**B.cfg)
    nsub = nsub_of(robot)
    for e, (task, sc, gap, robot_only, bogus) in enumerate(cases):
        o = orc[e]
        if sc[0] == "keep":   # the body stays where the reset put it and gets a velocity
            slot = [s for s, t in enumerate(o.slot_types()) if t == sc[1]][0]
            o.set_obj(slot, vx=sc[2][0], vy=sc[2][1], w=sc[2][2])
            continue
        scene = teleport(robot, cfg) if sc[0] == "teleport" else face(robot, sc[1], cfg, body_v=sc[2])
        if gap == "overlap":
            gap = bisect_gap(B.fresh_oracle(e), scene, None, nsub) - 1e-3
        scene(o, gap)
    for o in orc:
        o.forward()
        assert o.error == 0
    for e, c in enumerate(cases):   # the scenes are what they claim to be
        if c[2] == "overlap":
            assert orc[e].contacts(), e
    # objects first: the teleported robot's environment changes with the robot field alone
    fields = fields_from_oracles(env, orc, ("objects", "robot") + (("robot_ext",) if robot == "car" else ()))
    f64, i32 = env.get_field("task_f64").cpu(), env.get_field("task_i32").cpu()
    edit = False
    for e, c in enumerate(cases):
        if c[4] == "clear":
            f64[7, e] = 1e30; edit = True
        elif c[4] == "movmask":
            i32[9, e] = 0; edit = True
    if route == "load_state_dict":
        sd = env.state_dict()
        for k, v in fields.items():
            sd["fields"][k] = v
        sd["fields"]["task_f64"], sd["fields"]["task_i32"] = f64, i32
        env.load_state_dict(sd)
    else:
        write_fields(env, fields, route)
        if edit:   # derived rows written last, bogus
            write_fields(env, {"task_f64": f64, "task_i32": i32}, route)
    acts = np.zeros((len(cases), 2))
    contacts = step_both(env, orc, acts, steps, route=route, tag=f"{robot} {route}")
    env.close()
    return contacts


@pytest.mark.parametrize("robot", ["point", "car"])
@pytest.mark.parametrize("route", ["set_field", "load_state_dict", "abi"])
def test_injected_state_is_stepped_with_fresh_caches_hostemu(robot, route):
    assert run_injection("hostemu", robot, route) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["point", "car"])
@pytest.mark.parametrize("route", ["set_field", "load_state_dict", "abi"])
def test_injected_state_is_stepped_with_fresh_caches_gpu(robot, route):
    assert run_injection("cuda", robot, route) > 0


# the identity: writing back every field of a state the kernels left changes no bit
def run_write_back_identity(backend):
    batches = []
    names = ["go_to_goal", "haul_box", "push_box", "press_buttons", "roll_rod", "dribble_ball", "collect", "catch_goal",
             "go_to_goal_motor", "unsupervised"]
    env = make_env(backend, len(names), names, 5, {"action_noise": 0.01})
    # environment 0: all ten vases stacked into one heap in front of the robot (common.run_overflow_case): a sticky
    # PhysicsError
    objs, rob = env.get_field("objects"), env.get_field("robot")
    rx, ry = float(rob[0, 0]), float(rob[1, 0])
    for k, s in enumerate(range(9, 19)):
        objs[0, s, 0], objs[1, s, 0], objs[2, s, 0] = rx + 0.16 + 0.03 * (k % 4), ry + 0.03 * (k // 4) - 0.03, 0.1 * k
    rob[2, 0], rob[3, 0] = 0.0, 0.5
    env.set_field("objects", objs); env.set_field("robot", rob)
    batches.append((env, [0]))
    batches.append((make_env(backend, 6, ["go_to_goal", "push_box", "haul_box"] * 2, 6, {"action_noise": 0.01}, robot="car",
                             max_episode_steps=70), []))
    batches.append((make_env(backend, 4, ["go_to_goal", "push_box"] * 2, 7, {"num_gremlins": 2, "action_noise": 0.01}), []))
    for env, heap in batches:
        g = torch.Generator(device=env.device); g.manual_seed(3)
        for t in range(200):
            act = torch.rand((env.num_envs, 2), device=env.device, generator=g) * 2 - 1
            act[heap, 0], act[heap, 1] = 1.0, 0.0
            env.step(act)
        before = {k: env.get_field(k).cpu() for k in env._FIELDS}
        if heap:   # the heap's PhysicsError: done, not reset (no time limit)
            assert int(before["flags"][0]) != 0
        for k in env._FIELDS:
            env.set_field(k, before[k])
        after = {k: env.get_field(k).cpu() for k in env._FIELDS}
        for k in env._FIELDS:
            assert before[k].numpy().tobytes() == after[k].numpy().tobytes(), (env.robot_name, k)
        env.close()


def test_write_back_of_an_unchanged_state_changes_nothing_hostemu():
    run_write_back_identity("hostemu")


@pytest.mark.gpu
def test_write_back_of_an_unchanged_state_changes_nothing_gpu():
    run_write_back_identity("cuda")


# ------------------------------------------------------------------------------------------------------------------
# (b) the quiet / near threshold, (c) the object-pair broad phase, (d) the HaulBox tendon
# ------------------------------------------------------------------------------------------------------------------
_terminal = {}


def robot_state(robot, task, action, scale=1.0):
    """an extreme robot state: the one a constant action reaches from rest, its velocity scaled by `scale` (injected)"""
    key = (robot, task, tuple(action))
    if key not in _terminal:
        _terminal[key] = terminal_state(robot, task, action)
    vb, w, ext = _terminal[key]
    return dict(vb=(scale * vb[0], scale * vb[1]), w=w, ext=ext)


def threshold_scenes(robot, variant):
    """(task, action, robot state, kind) per scene"""
    if robot == "point":
        states = [("go_to_goal", (1.0, 0.0), 1.0), ("go_to_goal", (1.0, 0.0), 2.5), ("go_to_goal", (0.0, 1.0), 1.0),
                  ("go_to_goal", (0.0, -1.0), 1.0)]
    else:
        states = [("go_to_goal", (-1.0, -1.0), 1.0), ("go_to_goal", (1.0, -1.0), 1.0), ("go_to_goal", (-1.0, -1.0), 2.5)]
    kinds = list(KIND_TASK)
    if variant == "sizes":   # kind_bound reads vases_size / pillars_size
        states, kinds = states[:1] + states[2:3], [O.VASE, O.PILLAR]
    out = []
    for (task, action, scale) in states:
        for kind in kinds:
            out.append((KIND_TASK[kind], action, robot_state(robot, task, action, scale), kind))
    if robot == "point" and variant == "default":   # travel_bound reads gear_x and damp_xy
        for task in ("go_to_goal_motor", "go_to_goal_damping"):
            for kind in (O.VASE, O.PILLAR):
                out.append((task, (1.0, 0.0), robot_state(robot, task, (1.0, 0.0)), kind))
    return out


def gaps_around(g):
    return [g - d for d in DELTAS[::-1]] + [g + d for d in DELTAS] + [g + 0.3]   # the last one well inside the quiet range


def run_edge_batch(backend, robot, scenes, config=None, steps=3):
    """scenes: (task, action, scene(o, gap), bisection keywords) each; every scene is run at the gaps around its
    oracle-bisected g* (gaps_around), one environment per gap, kernel and oracle from the same injected state"""
    ng = len(gaps_around(0.0))
    tasks = [sc[0] for sc in scenes for _ in range(ng)]
    B = Batch(backend, robot, tasks, config)
    nsub = nsub_of(robot)
    acts = np.zeros((len(tasks), 2))
    first_hit = []
    for i, (task, action, scene, kw) in enumerate(scenes):
        e0 = i * ng
        g = bisect_gap(B.fresh_oracle(e0), scene, action, nsub, **kw)
        for k, gap in enumerate(gaps_around(g)):
            scene(B.orc[e0 + k], gap)
            acts[e0 + k] = action
        first_hit.append(e0)
    for o in B.orc:
        o.forward()
    write_fields(B.env, fields_from_oracles(B.env, B.orc, ("objects", "robot") + (("robot_ext",) if robot == "car" else ())), "set_field")
    obs = B.env.observation.cpu().numpy()
    for e, o in enumerate(B.orc):
        np.testing.assert_array_equal(obs[e], o.observation().astype(np.float32), err_msg=f"injected state env {e}")
    o0 = oracle_state(B.orc)[1]
    contacts = step_both(B.env, B.orc, acts, steps, tag=robot)
    B.env.close()
    moved = np.abs(oracle_state(B.orc)[1][:, :, :2] - o0[:, :, :2]).max(axis=(1, 2))
    return contacts, moved


def _threshold(backend, robot, variant):
    config = {"vases_size": 0.13, "pillars_size": 0.27} if variant == "sizes" else None
    cfg = O.default_config(**(config or {}))
    scenes = [(task, action, face(robot, kind, cfg, vb=st["vb"], w=st["w"], ext=st["ext"]), {})
              for task, action, st, kind in threshold_scenes(robot, variant)]
    assert run_edge_batch(backend, robot, scenes, config)[0] > 0


@pytest.mark.parametrize("robot,variant", [("point", "default"), ("point", "sizes"), ("car", "default")])
def test_quiet_near_threshold_hostemu(robot, variant):
    _threshold("hostemu", robot, variant)


@pytest.mark.gpu
@pytest.mark.parametrize("robot,variant", [("point", "default"), ("point", "sizes"), ("car", "default")])
def test_quiet_near_threshold_gpu(robot, variant):
    _threshold("cuda", robot, variant)


def pushed_into(robot, kind, other, cfg, st):
    """Scene: the robot at full speed 5 mm from a task body (corner first) that already slides away from it at 0.5 m/s,
    a resting vase / pillar beyond that body on the centre line, `gap` from it (farthest points facing)"""
    push = face(robot, kind, cfg, vb=st["vb"], w=st["w"], ext=st["ext"], body_v=(0.5, 0.0, 0.0))
    bf, ba = body_far(kind, cfg)
    of, oa = body_far(other, cfg)

    def scene(o, gap):
        push(o, 0.005)
        types = o.slot_types()
        slot = types.index(kind)
        ob = o.get_obj(slot)
        d = bf + of + gap
        s2 = types.index(other)
        o.set_obj(s2, x=ob.x + d * np.cos(PHI), y=ob.y + d * np.sin(PHI), yaw=PHI + np.pi - oa, vx=0.0, vy=0.0, w=0.0)
        _clear_others(o, {slot, s2}, o.robot_state[:2])
    return scene


def _object_pairs(backend, robot):
    cfg = O.default_config()
    action = (1.0, 0.0) if robot == "point" else (-1.0, -1.0)
    st = robot_state(robot, "go_to_goal", action)
    scenes = []
    for kind in (O.BOX, O.ROD, O.BALL):
        task = KIND_TASK[kind]
        slots = O.task_slot_types(task)
        for other in (O.VASE, O.PILLAR):
            if other not in slots:
                continue
            scenes.append((task, action, pushed_into(robot, kind, other, cfg, st), {"steps": 4, "pair": (slots.index(kind), slots.index(other))}))
    assert len(scenes) >= 3
    assert run_edge_batch(backend, robot, scenes, steps=6)[0] > 0


@pytest.mark.parametrize("robot", ["point", "car"])
def test_object_pair_broad_phase_hostemu(robot):
    _object_pairs("hostemu", robot)


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["point", "car"])
def test_object_pair_broad_phase_gpu(robot):
    _object_pairs("cuda", robot)


def hauled(robot, st):
    """Scene (HaulBox): the robot at full speed straight away from the box; `gap` is the tendon's slack, 0.75 minus the
    centre distance"""
    def scene(o, gap):
        rs = o.robot_state
        rs[2] = PHI + (0.0 if robot == "point" else np.pi / 2)   # heading (the car drives along body -y) = PHI
        sign = 1.0 if robot == "point" else -1.0
        rs[3], rs[4] = _rot((st["vb"][0], sign * abs(st["vb"][1])) if robot == "point" else st["vb"], rs[2])
        rs[5] = st["w"]
        o.robot_state = rs
        if robot == "car":
            o.robot_ext = st["ext"]
        slot = o.slot_types().index(O.BOX)
        d = 0.75 - gap
        o.set_obj(slot, x=rs[0] - d * np.cos(PHI), y=rs[1] - d * np.sin(PHI), yaw=0.0, vx=0.0, vy=0.0, w=0.0)
        _clear_others(o, {slot}, rs[:2])
    return scene


def _tendon(backend, robot):
    action = (1.0, 0.0) if robot == "point" else (1.0, 1.0)
    st = robot_state(robot, "go_to_goal", action)
    slot = O.task_slot_types("haul_box").index(O.BOX)
    scenes = [("haul_box", action, hauled(robot, st), {"moved": slot, "lo": -0.3, "hi": 0.3})]
    _, moved = run_edge_batch(backend, robot, scenes, steps=3)
    assert (moved[:len(DELTAS)] > 0).all() and moved[-1] == 0.0, moved   # pulled inside g*, at rest well outside it


@pytest.mark.parametrize("robot", ["point"])
def test_haul_box_tendon_slack_hostemu(robot):
    _tendon("hostemu", robot)


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["point"])
def test_haul_box_tendon_slack_gpu(robot):
    _tendon("cuda", robot)
