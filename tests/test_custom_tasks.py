"""User-defined tasks: Task subclasses with their own obstacle counts and placement extents, run on the device path
bit for bit against oracle environments built from the same descriptor (tests/oracle_spec: orc_env_create_spec).

Every case runs on the CPU against the host emulation of tests/hostemu/sag_hostemu_custom.cpp (the *C instantiations
of the kernel body) and, marked gpu, on the CUDA library."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import oracle as O
from safe_adaptation_gym_b200 import _abi, tasks
from safe_adaptation_gym_b200.env import BatchedSafeAdaptationGym
from safe_adaptation_gym_b200.utils import ResamplingError

from common import drive_action, env_state, oracle_state

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOSTEMU_LIB = os.path.join(ROOT, "tests", "hostemu", "libsag_hostemu_custom.so")
SPEC_LIB = os.path.join(ROOT, "tests", "oracle_spec", "libsag_oracle_spec.so")
FMA = ["-mfma"] if "fma" in open("/proc/cpuinfo").read().split() else []
_libs = {}


def hostemu_lib():
    if "hostemu" not in _libs:
        if not os.path.exists(HOSTEMU_LIB):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off"] + FMA +
                                  ["-o", HOSTEMU_LIB, HOSTEMU_LIB.replace("libsag_hostemu_custom.so", "sag_hostemu_custom.cpp")])
        _libs["hostemu"] = _abi.SagLib(HOSTEMU_LIB, host_api=False)
    return _libs["hostemu"]


def spec_lib():
    """the oracle with orc_env_create_spec; the prototypes are the oracle's own"""
    if "spec" not in _libs:
        if not os.path.exists(SPEC_LIB):
            subprocess.check_call(["gcc", "-O2", "-std=gnu99", "-fPIC", "-ffp-contract=off", "-pthread", "-shared"] + FMA +
                                  ["-o", SPEC_LIB, SPEC_LIB.replace("libsag_oracle_spec.so", "sag_oracle_spec.c"), "-lm"])
        L, ref = C.CDLL(SPEC_LIB), O.lib()
        for name in dir(ref):
            if name.startswith("orc_"):
                f, g = getattr(ref, name), getattr(L, name)
                g.argtypes, g.restype = f.argtypes, f.restype
        L.orc_env_create_spec.restype = C.c_void_p
        L.orc_env_create_spec.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(O.Config)]
        _libs["spec"] = L
    return _libs["spec"]


class SpecOracle(O.OracleEnv):
    """An oracle environment of a user-defined task (or of a registry task: its own descriptor)"""

    def __init__(self, robot, task, config=None, seed=0, env_gid=0):
        base, obstacles, extents = tasks.definition(task)
        self.L = spec_lib()
        self.cfg = O.Config()
        self.L.orc_default_config(C.byref(self.cfg))
        for k, v in (config or {}).items():
            if hasattr(self.cfg, k):
                setattr(self.cfg, k, v)
        self.robot = {"point": O.POINT, "car": O.CAR}[robot]
        self.task = base.task_id
        self.h = self.L.orc_env_create_spec(self.robot, base.task_id, (C.c_int * 4)(*obstacles),
                                            (C.c_double * 4)(*extents), C.byref(self.cfg))
        assert self.h
        self.L.orc_env_seed(self.h, seed, env_gid)
        self._replay = None


def custom(base, obstacles=None, extents=None, name=None):
    """a Task subclass of `base` overriding obstacles and / or placement_extents"""
    body = {}
    if obstacles is not None:
        body["obstacles"] = property(lambda self: list(obstacles))
    if extents is not None:
        body["placement_extents"] = property(lambda self: tuple(extents))
    return type(name or "Custom" + base.__name__, (base,), body)


def make(backend, n, task_list, seed, config=None, robot="point", **kw):
    cfg = dict(config or {})
    cfg.setdefault("action_noise", 0.0)
    lib = hostemu_lib() if backend == "hostemu" else None
    env = BatchedSafeAdaptationGym("xmls/%s.xml" % robot, config=cfg, num_envs=n, _test_lib=lib, **kw)
    env.seed(seed)
    if task_list is not None:
        env.set_task(task_list)
    return env


def oracles(task_list, seed, config=None, robot="point", gid_base=0):
    cfg = dict(config or {})
    cfg.setdefault("action_noise", 0.0)
    envs = [SpecOracle(robot, t, cfg, seed, gid_base + e) for e, t in enumerate(task_list)]
    for e in envs:
        assert e.reset(0) == 0
    return envs


def used_slots(o, orc):
    """the object slots the oracle environments use (a task switch leaves the device's other slots as they were)"""
    o = o.copy()
    for e, oe in enumerate(orc):
        o[e, oe.nobj:] = 0.0
    return o


def compare(env, orc, steps, seed, check_every=1):
    """bit-exact layout, then per step observation, reward, cost and done (and the state every check_every steps)"""
    r, o = env_state(env)
    ro, oo = oracle_state(orc)
    np.testing.assert_array_equal(r, ro)
    np.testing.assert_array_equal(used_slots(o, orc), oo)
    rng = np.random.RandomState(seed + 17)
    n = len(orc)
    events = {"cost": 0.0, "contacts": 0}
    for t in range(steps):
        acts = np.stack([drive_action(orc[e], rng) for e in range(n)]).astype(np.float32)
        obs, rew, done, info = env.step(torch.from_numpy(acts).to(env.device))
        obs, rew = obs.cpu().numpy(), rew.cpu().numpy()
        cost, done = info["cost"].cpu().numpy(), done.cpu().numpy()
        for e in range(n):
            oobs, orew, ocost, odone, rc = orc[e].step(acts[e].astype(np.float64))
            assert rc == 0
            np.testing.assert_array_equal(obs[e], oobs.astype(np.float32), err_msg=f"env {e} step {t}")
            r = rew[e] if rew.ndim == 2 else rew[e:e + 1]   # Unsupervised: the reward pair
            np.testing.assert_array_equal(r, orew[:len(r)], err_msg=f"env {e} step {t}")
            assert cost[e] == ocost and bool(done[e]) == odone, f"env {e} step {t}"
            events["cost"] += ocost
            events["contacts"] += len(orc[e].contacts())
        if (t + 1) % check_every == 0:
            r, o = env_state(env)
            ro, oo = oracle_state(orc)
            np.testing.assert_array_equal(r, ro, err_msg=f"step {t}")
            np.testing.assert_array_equal(used_slots(o, orc), oo, err_msg=f"step {t}")
    return events


BASES = [tasks.GoToGoal, tasks.PressButtons, tasks.Collect, tasks.PushBox, tasks.HaulBox, tasks.CatchGoal,
         tasks.Unsupervised]


def base_task_objects(base):
    return base.NUM_BUTTONS if issubclass(base, tasks.PressButtons) else 2 if issubclass(base, tasks.PushBox) else 1


def case_task(base, case):
    if case == "zero_hazards":
        return custom(base, obstacles=[0] + list(base().obstacles[1:]))
    if case == "full":  # all 32 slots (a box base puts its box in slot 31); small keepouts so that the layout can be sampled
        free = 32 - base_task_objects(base)
        return custom(base, obstacles=[free - 12, 10, 0, 2], extents=(-3.5, -3.5, 3.5, 3.5))
    if case == "asymmetric":
        return custom(base, obstacles=[3, 2, 0, 1], extents=(-1.5, -3.0, 2.5, 1.0))
    if case == "gremlins":
        return custom(base, obstacles=[4, 3, 2, 1], extents=(-2.5, -2.0, 2.5, 2.0))
    raise ValueError(case)


FULL_CFG = {"hazards_keepout": 0.18, "vases_keepout": 0.1, "pillars_keepout": 0.2}


def run_trajectories(backend, robot, base, case, n=3, steps=300, seed=31):
    cfg = dict(FULL_CFG) if case == "full" else {}
    if case == "gremlins":
        cfg["num_gremlins"] = 2
    cls = case_task(base, case)
    tl = [cls()] * n
    env = make(backend, n, tl, seed, cfg, robot=robot)
    assert env.task_id_of(cls()) == _abi.NUM_TASKS
    assert env.task_ids.cpu().tolist() == [_abi.NUM_TASKS] * n
    compare(env, oracles(tl, seed, cfg, robot=robot), steps, seed, check_every=50)


@pytest.mark.parametrize("robot", ["point", "car"])
@pytest.mark.parametrize("base", BASES, ids=lambda c: c.name)
@pytest.mark.parametrize("case", ["zero_hazards", "full", "asymmetric", "gremlins"])
def test_trajectories_vs_oracle_hostemu(robot, base, case):
    run_trajectories("hostemu", robot, base, case, steps=300 if robot == "point" else 120)


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["point", "car"])
@pytest.mark.parametrize("base", BASES, ids=lambda c: c.name)
@pytest.mark.parametrize("case", ["zero_hazards", "full", "asymmetric", "gremlins"])
def test_trajectories_vs_oracle_gpu(robot, base, case):
    run_trajectories("cuda", robot, base, case, n=8)


def run_equal_spec(backend, seed=41):
    Same = custom(tasks.PushBox, obstacles=[2, 3, 0, 1], extents=(-1.75, -1.75, 1.75, 1.75), name="SamePushBox")
    a = make(backend, 4, [Same()] * 4, seed)
    b = make(backend, 4, [tasks.PushBox()] * 4, seed)
    assert a.task_id_of(Same()) == tasks.PushBox.task_id and a._custom == []
    assert a.task_stats().shape == (14, 3)
    rng = np.random.RandomState(0)
    for _ in range(60):
        act = torch.from_numpy(rng.uniform(-1, 1, (4, 2)).astype(np.float32)).to(a.device)
        oa, ra, da, ia = a.step(act)
        ob, rb, db, ib = b.step(act)
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(ia["cost"], ib["cost"])
    for f in ("robot", "objects", "task_f64", "task_i32"):
        assert torch.equal(a.get_field(f), b.get_field(f))


def test_equal_spec_keeps_base_id_hostemu():
    run_equal_spec("hostemu")


@pytest.mark.gpu
def test_equal_spec_keeps_base_id_gpu():
    run_equal_spec("cuda")


def define_raw(env, base, obstacles, extents):
    d = _abi.SagTaskDef(base.task_id, (C.c_int32 * 4)(*obstacles), (C.c_double * 4)(*extents))
    tid = C.c_int32()
    env._lib.check(env._lib.L.sag_define_task(env._h, C.byref(d), C.byref(tid)))
    return tid.value


def run_custom_id_with_base_values(backend, seed=43, n=4, max_steps=40):
    """A custom id carrying the base's values runs bit-identically to the base; its statistics have their own row"""
    a = make(backend, n, [tasks.GoToGoal()] * n, seed, max_episode_steps=max_steps)
    b = make(backend, n, [tasks.GoToGoal()] * n, seed, max_episode_steps=max_steps)
    tid = define_raw(a, tasks.GoToGoal, [9, 10, 0, 1], [-2, -2, 2, 2])
    assert tid == 14 and a._lib.L.sag_num_task_ids(a._h) == 15
    ids = torch.full((n,), tid, dtype=torch.int32, device=a.device)
    a._lib.check(a._lib.L.sag_set_tasks(a._h, a._p(ids), a._stream()))
    a._reset_all(new_task=True)
    b.set_task([tasks.GoToGoal()] * n)   # the same second reset (episode 1, fresh task instances)
    rng = np.random.RandomState(1)
    for _ in range(2 * max_steps + 5):
        act = torch.from_numpy(rng.uniform(-1, 1, (n, 2)).astype(np.float32)).to(a.device)
        oa, ra, da, ia = a.step(act)
        ob, rb, db, ib = b.step(act)
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
    out = torch.zeros((15, 3), dtype=torch.float64, device=a.device)
    a._lib.check(a._lib.L.sag_task_stats(a._h, a._p(out), 0, a._stream()))
    sb = b.task_stats()
    assert torch.equal(out[14], sb[3]) and float(out[14, 2]) == 2 * n and float(out[3, 2]) == 0.0


def test_custom_id_with_base_values_hostemu():
    run_custom_id_with_base_values("hostemu")


@pytest.mark.gpu
def test_custom_id_with_base_values_gpu():
    run_custom_id_with_base_values("cuda")


FewHazards = custom(tasks.GoToGoal, obstacles=[4, 10, 0, 1], name="FewHazards")
Cramped = custom(tasks.PushBox, extents=(-1.5, -1.25, 1.5, 1.25), name="Cramped")


def run_mixed_and_switches(backend, seed=51, n=6, max_steps=25):
    """registry and custom tasks in one batch; set_task with a mask; set_next_task into and out of custom tasks,
    checked against oracle environments built for each environment's task and episode"""
    tl = [tasks.GoToGoal(), FewHazards(), tasks.PushBox(), Cramped(), FewHazards(), tasks.GoToGoal()]
    env = make(backend, n, tl, seed, max_episode_steps=max_steps)
    assert env.task_ids.cpu().tolist() == [3, 14, 10, 15, 14, 3]
    compare(env, oracles(tl, seed), 10, seed)
    # queue: every env switches at its next reset, the auto-reset at the time limit (step 25 of episode 0)
    nxt = [tasks.GoToGoal(), tasks.PushBox(), Cramped(), FewHazards(), Cramped(), FewHazards()]
    env.set_next_task(nxt)
    before = env.task_ids.cpu().tolist()
    rng = np.random.RandomState(3)
    for _ in range(max_steps - 10):
        env.step(torch.from_numpy(rng.uniform(-1, 1, (n, 2)).astype(np.float32)).to(env.device))
    assert env.task_ids.cpu().tolist() == [env.task_id_of(t) for t in nxt]
    stats = env.task_stats()
    assert stats.shape == (16, 3)
    counts = {i: float(stats[i, 2]) for i in range(16) if stats[i, 2] > 0}
    expect = {}
    for t in before:   # the finished episodes count under the tasks they ran
        expect[t] = expect.get(t, 0.0) + 1.0
    assert counts == expect

    def fresh_oracles(task_list, envs_idx):
        orc = []
        for e in envs_idx:
            o = SpecOracle("point", task_list[e], {"action_noise": 0.0}, seed, e)
            assert o.reset(int(env.get_field("task_i32")[8, e])) == 0
            orc.append(o)
        return orc

    orc = fresh_oracles(nxt, range(n))
    r, o = env_state(env)
    ro, oo = oracle_state(orc)
    np.testing.assert_array_equal(r, ro)
    np.testing.assert_array_equal(used_slots(o, orc), oo)
    compare(env, orc, 10, seed + 1)
    # mask: envs 0 and 2 switch now, into and out of custom tasks
    new = list(nxt)
    new[0], new[2] = FewHazards(), tasks.GoToGoal()
    env.set_task(new, mask=[True, False, True, False, False, False])
    assert env.task_ids.cpu().tolist() == [env.task_id_of(t) for t in new]
    r, o = env_state(env)
    orc = fresh_oracles(new, [0, 2])
    ro, oo = oracle_state(orc)
    np.testing.assert_array_equal(r[[0, 2]], ro)
    np.testing.assert_array_equal(used_slots(o[[0, 2]], orc), oo)


def test_mixed_and_switches_hostemu():
    run_mixed_and_switches("hostemu")


@pytest.mark.gpu
def test_mixed_and_switches_gpu():
    run_mixed_and_switches("cuda")


def run_copy_envs(backend, seed=61, n=4):
    a = make(backend, n, [FewHazards(), tasks.GoToGoal(), FewHazards(), Cramped()], seed)
    b = make(backend, n, [FewHazards(), tasks.GoToGoal(), FewHazards(), Cramped()], seed + 1)
    b.copy_envs([3, 2, 1, 0], source=a)
    for f in ("robot", "objects", "task_i32"):
        assert torch.equal(b.get_field(f)[..., :n], a.get_field(f)[..., [3, 2, 1, 0]])
    c = make(backend, n, [Cramped(), FewHazards(), Cramped(), Cramped()], seed)   # other definition order
    with pytest.raises(ValueError, match="user-defined tasks"):
        c.copy_envs([0, 1, 2, 3], source=a)
    L = a._lib
    idx = torch.arange(n, dtype=torch.int32, device=a.device)
    with pytest.raises(_abi.SagError, match="user-defined tasks"):
        L.check(L.L.sag_copy_envs(c._h, a._h, c._p(idx), c._stream()))


def test_copy_envs_hostemu():
    run_copy_envs("hostemu")


@pytest.mark.gpu
def test_copy_envs_gpu():
    run_copy_envs("cuda")


def run_evaluate_actions(backend, seed=71, n=4, H=6):
    tl = [FewHazards(), Cramped(), tasks.GoToGoal(), FewHazards()]
    a = make(backend, n, tl, seed)
    b = make(backend, n, tl, seed)
    acts = torch.from_numpy(np.random.RandomState(5).uniform(-1, 1, (H, n, 2)).astype(np.float32)).to(a.device)
    obs, ret, cost, length = a.evaluate_actions(acts)
    r = torch.zeros(n, dtype=torch.float64, device=b.device)
    c = torch.zeros(n, dtype=torch.float64, device=b.device)
    ln = torch.zeros(n, dtype=torch.int32, device=b.device)
    live = torch.ones(n, dtype=torch.bool, device=b.device)
    for h in range(H):   # the sums stop at the first done (a physics error)
        ob, rb, db, ib = b.step(acts[h])
        r += torch.where(live, rb, 0.0)
        c += torch.where(live, ib["cost"].to(torch.float64), 0.0)
        ln += live.to(torch.int32)
        live &= ~db
    assert torch.equal(obs, ob) and torch.equal(ret, r) and torch.equal(cost, c) and torch.equal(length, ln)
    for f in ("robot", "objects", "task_f64", "task_i32"):
        assert torch.equal(a.get_field(f), b.get_field(f))


def test_evaluate_actions_hostemu():
    run_evaluate_actions("hostemu")


@pytest.mark.gpu
def test_evaluate_actions_gpu():
    run_evaluate_actions("cuda")


def run_state_dict(backend, seed=81, n=4):
    tl = [FewHazards(), Cramped(), tasks.GoToGoal(), Cramped()]
    a = make(backend, n, tl, seed)
    rng = np.random.RandomState(2)
    acts = [torch.from_numpy(rng.uniform(-1, 1, (n, 2)).astype(np.float32)).to(a.device) for _ in range(30)]
    for t in acts[:10]:
        a.step(t)
    sd = a.state_dict()
    b = make(backend, n, None, seed + 5)
    b.load_state_dict(sd)
    assert b._definitions() == a._definitions() and b.task_ids.tolist() == a.task_ids.tolist()
    # the user's classes take the restored ids: no second definition, the statistics keep their shape
    assert [b.task_id_of(t) for t in (FewHazards(), Cramped())] == [14, 15]
    assert b._definitions() == a._definitions() and b.task_stats().shape == a.task_stats().shape == (16, 3)
    for t in acts[10:20]:
        oa, ra, _, _ = a.step(t)
        ob, rb, _, _ = b.step(t)
        assert torch.equal(oa, ob) and torch.equal(ra, rb)
    a.set_next_task([Cramped(), FewHazards(), None, FewHazards()])
    b.set_next_task([Cramped(), FewHazards(), None, FewHazards()])
    a.reset()
    b.reset()
    assert a.task_ids.tolist() == b.task_ids.tolist() == [15, 14, 3, 14]
    for t in acts[20:]:
        oa, ra, _, _ = a.step(t)
        ob, rb, _, _ = b.step(t)
        assert torch.equal(oa, ob) and torch.equal(ra, rb)
    b.copy_envs([0, 1, 2, 3], source=a)   # the tables still agree
    c = make(backend, n, [Cramped()] * n, seed)   # defines Cramped first: conflicts
    with pytest.raises(ValueError, match="conflict"):
        c.load_state_dict(sd)


def test_state_dict_hostemu():
    run_state_dict("hostemu")


@pytest.mark.gpu
def test_state_dict_gpu():
    run_state_dict("cuda")


def run_refusals(backend, monkeypatch):
    env = make(backend, 2, [tasks.GoToGoal()] * 2, 1)

    class BigGoal(tasks.GoToGoal):
        GOAL_SIZE = 0.5

    class OwnReward(tasks.GoToGoal):
        def compute_reward(self, *a):
            return 0.0

    with pytest.raises(NotImplementedError, match="GOAL_SIZE"):
        env.set_task(BigGoal())
    with pytest.raises(NotImplementedError, match="compute_reward"):
        env.task_id_of(OwnReward())
    for obstacles, extents, match in (([-1, 10, 0, 1], None, ">= 0"), ([20, 11, 0, 1], None, "slots"),
                                      ([9, 10, 1, 1], None, "num_gremlins"), (None, (2, -2, -2, 2), "x_min"),
                                      (None, (-2, 2, 2, -2), "y_min")):
        with pytest.raises(ValueError, match=match):
            env.set_task(custom(tasks.GoToGoal, obstacles, extents)())
    assert env._custom == [] and env._lib.L.sag_num_task_ids(env._h) == 14
    # the library validates too
    for obstacles, extents in (([9, 10, 0, 1], [2, -2, -2, 2]), ([31, 1, 0, 1], [-2, -2, 2, 2]), ([9, 10, 1, 1], [-2, -2, 2, 2])):
        with pytest.raises(_abi.SagError):
            define_raw(env, tasks.GoToGoal, obstacles, extents)
    for k in range(16):
        env.task_id_of(custom(tasks.GoToGoal, obstacles=[k, 1, 0, 0])())
    with pytest.raises(ValueError, match="at most 16"):
        env.task_id_of(custom(tasks.GoToGoal, obstacles=[1, 2, 0, 0])())
    with pytest.raises(_abi.SagError):
        define_raw(env, tasks.GoToGoal, [1, 2, 0, 0], [-2, -2, 2, 2])
    # a layout that cannot be sampled
    tight = make(backend, 2, [tasks.GoToGoal()] * 2, 1, {"max_layout_draws": 20000})
    with pytest.raises(ResamplingError):
        tight.set_task(custom(tasks.GoToGoal, extents=(-0.8, -0.8, 0.8, 0.8))())
    # definitions under capture
    import safe_adaptation_gym_b200.env as E
    fresh = make(backend, 2, [tasks.GoToGoal()] * 2, 1)
    monkeypatch.setattr(E, "_capturing", lambda: True)
    with pytest.raises(RuntimeError, match="capture"):
        fresh.task_id_of(FewHazards())


def test_refusals_hostemu(monkeypatch):
    run_refusals("hostemu", monkeypatch)


@pytest.mark.gpu
def test_refusals_gpu(monkeypatch):
    run_refusals("cuda", monkeypatch)


def run_reset_options(backend, seed=83, n=3):
    """reset(options={'task': ...}) with user-defined tasks, against the oracle"""
    env = make(backend, n, [tasks.GoToGoal()] * n, seed)
    tl = [FewHazards(), Cramped(), FewHazards()]
    env.reset(options={"task": tl})
    assert env.task_ids.tolist() == [14, 15, 14]
    orc = []
    for e, t in enumerate(tl):
        o = SpecOracle("point", t, {"action_noise": 0.0}, seed, e)
        assert o.reset(int(env.get_field("task_i32")[8, e])) == 0
        orc.append(o)
    compare(env, orc, 40, seed)


def test_reset_options_hostemu():
    run_reset_options("hostemu")


@pytest.mark.gpu
def test_reset_options_gpu():
    run_reset_options("cuda")


def test_tasks_defined_through_the_c_abi_count_in_task_stats_hostemu():
    env = make("hostemu", 2, [tasks.GoToGoal()] * 2, 1)
    define_raw(env, tasks.GoToGoal, [9, 10, 0, 1], [-2, -2, 2, 2])
    assert env.task_stats().shape == (15, 3)


@pytest.mark.parametrize("robot", ["point", "car"])
@pytest.mark.parametrize("task", ["go_to_goal_damping", "press_buttons_scarce", "collect", "push_box_scarce", "haul_box",
                                  "roll_rod", "dribble_ball", "catch_goal", "unsupervised"])
def test_spec_oracle_of_a_registry_task_is_the_oracle(robot, task):
    """orc_env_create_spec restates the oracle's reset with the descriptor's slots: for a registry task's own descriptor
    it must be the oracle, draw for draw (so a change to the oracle's reset that the restatement misses fails here)"""
    from safe_adaptation_gym_b200.benchmark import TASKS
    seed, cfg = 57, {"action_noise": 0.0}
    for ng in (0, 2):
        c = dict(cfg, num_gremlins=ng)
        t = TASKS[task]()
        spec = custom(type(t), obstacles=list(t.obstacles[:2]) + [ng, t.obstacles[3]], name="Spec")()
        for gid in range(3):
            a, b = O.OracleEnv(robot, task, config=c, seed=seed, env_gid=gid), SpecOracle(robot, spec, c, seed, gid)
            for episode in (0, 1):
                assert a.reset(episode) == b.reset(episode) == 0
                np.testing.assert_array_equal(a.robot_state, b.robot_state)
                np.testing.assert_array_equal(a.objects(), b.objects())
                rng = np.random.RandomState(gid)
                for _ in range(60):
                    act = rng.uniform(-1, 1, 2)
                    ra, rb = a.step(act), b.step(act)
                    np.testing.assert_array_equal(ra[0], rb[0])
                    np.testing.assert_array_equal(ra[1], rb[1])
                    assert ra[2:] == rb[2:]


def test_unsupervised_custom_records_pair_hostemu():
    U = custom(tasks.Unsupervised, obstacles=[2, 2, 0, 1], name="SmallUnsupervised")
    env = make("hostemu", 2, [U(), tasks.GoToGoal()], 3)
    assert env._any_unsupervised
    _, rew, _, _ = env.step(torch.zeros((2, 2)))
    assert tuple(rew.shape) == (2, 2)
    g = make("hostemu", 2, [tasks.GoToGoal()] * 2, 3)
    with pytest.raises(ValueError, match="pair"):
        g.set_next_task([U(), None])


@pytest.mark.gpu
def test_large_batch_sampled_vs_oracle_gpu():
    """65,536 point environments, half GoToGoal and half a GoToGoal with 15 hazards and 6 vases; 256 sampled
    environments against the oracle every 50 steps"""
    n, seed, steps = 65536, 91, 300
    Hard = custom(tasks.GoToGoal, obstacles=[15, 6, 0, 1], name="Hard")
    tl = [tasks.GoToGoal() if e % 2 == 0 else Hard() for e in range(n)]
    env = make("cuda", n, tl, seed)
    pick = np.random.RandomState(0).choice(n, 256, replace=False)
    orc = [SpecOracle("point", tl[e], {"action_noise": 0.0}, seed, int(e)) for e in pick]
    for o in orc:
        assert o.reset(0) == 0
    rng = np.random.RandomState(4)
    for t in range(steps):
        acts = rng.uniform(-1, 1, (n, 2)).astype(np.float32)
        obs, rew, done, info = env.step(torch.from_numpy(acts).cuda())
        for k, e in enumerate(pick):
            oobs, orew, ocost, odone, rc = orc[k].step(acts[e].astype(np.float64))
            if (t + 1) % 50 == 0:
                assert float(rew[e]) == orew[0] and float(info["cost"][e]) == ocost
                np.testing.assert_array_equal(obs[e].cpu().numpy(), oobs.astype(np.float32))
        if (t + 1) % 50 == 0:
            r, o = env_state(env)
            ro, oo = oracle_state(orc)
            np.testing.assert_array_equal(r[pick], ro)
            np.testing.assert_array_equal(used_slots(o[pick], orc), oo)


@pytest.mark.gpu
def test_graphed_schedule_with_custom_ids_gpu():
    """policy + step + set_next_task as one CUDA graph, walking a schedule with custom ids, bit-identical to eager"""
    n, seed, T = 1024, 93, 40
    sched = [FewHazards(), tasks.GoToGoal(), Cramped(), tasks.PushBox()]
    envs = [make("cuda", n, [tasks.GoToGoal()] * n, seed, max_episode_steps=15) for _ in range(2)]
    ids = [envs[0].task_id_of(t) for t in sched]
    assert [envs[1].task_id_of(t) for t in sched] == ids == [14, 3, 15, 10]
    ids = torch.tensor(ids, dtype=torch.int32, device="cuda")
    W = torch.from_numpy(np.random.RandomState(0).normal(size=(60, 2)).astype(np.float32) * 0.1).cuda()
    k = torch.zeros((), dtype=torch.int64, device="cuda")

    def body(env, obs):
        nxt = ids[(k + torch.arange(n, device="cuda")) % len(sched)].to(torch.int32)
        env.set_next_task(nxt)
        out = env.step(torch.tanh(obs[:, :60] @ W))
        k.add_(1)
        return out

    eager, graphed = envs
    obs_e = eager.observation.clone()
    static_obs = graphed.observation.clone()
    k0 = k.clone()
    warm = make("cuda", n, [tasks.GoToGoal()] * n, seed, max_episode_steps=15)   # warm-up on a third batch
    assert [warm.task_id_of(t) for t in sched] == ids.tolist()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            body(warm, warm.observation)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out_g = body(graphed, static_obs)
    for t in range(T):
        k.copy_(k0 + t)
        out_e = body(eager, obs_e)
        obs_e = out_e[0].clone()
        k.copy_(k0 + t)
        g.replay()
        static_obs.copy_(out_g[0])
        assert torch.equal(out_e[0], out_g[0]) and torch.equal(out_e[1], out_g[1])
    assert torch.equal(eager.task_ids, graphed.task_ids)
    se, sg = eager.task_stats(), graphed.task_stats()
    assert se.shape == (16, 3) and torch.equal(se[:, 2], sg[:, 2])   # the sums are atomics: their order may differ
    torch.testing.assert_close(se, sg, rtol=1e-12, atol=1e-9)
