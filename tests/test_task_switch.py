"""Per-environment task switches at episode boundaries (env.set_next_task, the SAG_F_NEXT_TASK slot consumed by every
reset path).  Each case runs on the host emulation with the slot (CPU, tests/hostemu/sag_hostemu_next_task.cpp) and
on the CUDA library (-m gpu): a switching environment must equal an oracle environment built for the new task, that
episode and a fresh Task instance, bit for bit; the environments without a queued task must equal a twin that never
queued anything."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import common
import oracle as O
from common import env_state, oracle_state
from safe_adaptation_gym_b200 import _abi, tasks
from safe_adaptation_gym_b200.benchmark import TASK_IDS, TASKS
from safe_adaptation_gym_b200.env import BatchedSafeAdaptationGym

HOSTEMU_SRC = os.path.join(common.ROOT, "tests", "hostemu", "sag_hostemu_next_task.cpp")
HOSTEMU_LIB = os.path.join(common.ROOT, "tests", "hostemu", "libsag_hostemu_next_task.so")
_hostemu = None


def hostemu_lib():
    """g++ build of the host emulation with the next-task slot (tests/hostemu/sag_hostemu_next_task.cpp)."""
    global _hostemu
    if _hostemu is None:
        deps = [HOSTEMU_SRC, common.HOSTEMU_SRC] + [os.path.join(common.ROOT, p) for p in (
            "safe_adaptation_gym_b200/csrc/sag_core.cuh", "safe_adaptation_gym_b200/csrc/sag_layout.h",
            "include/sag_b200.h", "include/sag_detmath.h")]
        if not os.path.exists(HOSTEMU_LIB) or os.path.getmtime(HOSTEMU_LIB) < max(os.path.getmtime(d) for d in deps):
            fma = ["-mfma"] if "fma" in open("/proc/cpuinfo").read().split() else []
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off"] + fma +
                                  ["-o", HOSTEMU_LIB, HOSTEMU_SRC])
        _hostemu = _abi.SagLib(HOSTEMU_LIB, host_api=False)
    return _hostemu


def make_env(backend, n, task_names, seed, config=None, robot="point", **kw):
    """common.make_env, with the host emulation that has the next-task slot for backend 'hostemu'."""
    if backend != "hostemu":
        return common.make_env(backend, n, task_names, seed, config, robot=robot, **kw)
    env = BatchedSafeAdaptationGym("xmls/%s.xml" % robot, config=config, num_envs=n, _test_lib=hostemu_lib(), **kw)
    env.seed(seed)
    if isinstance(task_names, str):
        task_names = [task_names] * n
    env.set_task([TASKS[t]() for t in task_names])
    return env

T = 7  # max_episode_steps of the short-episode cases
MIXED = ["go_to_goal", "press_buttons", "push_box", "collect", "catch_goal", "haul_box", "go_to_goal_scarce", "roll_rod"]
CFG = {"action_noise": 0.0, "random_bound": True, "robot_ctrl_range_scale": 0.3}


def _dev(env):
    return "cuda" if env.device.type == "cuda" else "cpu"


def _stagger(envs, offsets):
    """Put the environments out of phase: environment e has already run offsets[e] steps of its episode."""
    for env in envs:
        ti = env.get_field("task_i32")
        ti[6, :env.num_envs] = torch.as_tensor(offsets, dtype=torch.int32, device=ti.device)
        env.set_field("task_i32", ti)


def _set_bodies_moving(envs):
    """A small velocity in every object slot (the same in every env), so that movable bodies are on the work list."""
    for env in envs:
        objs = env.get_field("objects")
        objs[3] = 0.2
        env.set_field("objects", objs)
        _ = env.observation


def _snap(out):
    obs, rew, done, info = out
    return [t.clone() for t in (obs, rew, done, info["cost"], info["bound"], info["truncated"])]


def _column(env, e):
    """State of environment e: robot [6] (+ 6 car extras), objects [32, 6], task_f64 [15], task_i32 [10]."""
    robot = env.get_field("robot")[:, e]
    if env.robot_name == "car":
        robot = torch.cat([robot, env.get_field("robot_ext")[:, e]])
    return (robot.cpu().numpy(), env.get_field("objects")[:, :, e].T.cpu().numpy(), env.get_field("task_f64")[:, e].cpu().numpy(),
            env.get_field("task_i32")[:, e].cpu().numpy())


def _check_fresh_instance(env, e, robot, cfg, seed):
    """State of environment e right after a switch == an oracle environment of its (new) task, its episode number and a
    fresh Task instance: robot, the task's objects, ctrl scales and bound (task_f64 rows 12-14), task id.  Returns the
    oracle."""
    r, objs, f64, i32 = _column(env, e)
    task, episode = int(i32[0]), int(i32[8])
    o = O.OracleEnv(robot, task, config=cfg, seed=seed, env_gid=env.env_id_base + e)
    o.new_task()
    assert o.reset(episode) == 0
    ro, oo = oracle_state([o])
    msg = f"env {e} (task {task}, episode {episode})"
    np.testing.assert_array_equal(r, ro[0], err_msg="robot of " + msg)
    # (the slots past the new task's objects are unused and keep what the previous task left there, as after set_task)
    np.testing.assert_array_equal(objs[:o.nobj], oo[0][:o.nobj], err_msg="objects of " + msg)
    np.testing.assert_array_equal(f64[12:14], o.ctrlrange[1], err_msg="ctrl scales of " + msg)
    assert f64[14] == o.bound, msg
    assert task == o.task, msg
    return o


# ---- the switch itself ------------------------------------------------------------------------------------------------
def run_switch_at_episode_ends(backend, n, names, robot="point", gremlins=0, moving=False, seed=11):
    """Queue tasks for a subset of an out-of-phase batch: only the queued environments switch, each exactly at its own
    episode end, and take the new task as a fresh Task instance; done / truncated and everything of the others is what a
    twin that queued nothing computes."""
    cfg = dict(CFG, num_gremlins=gremlins) if gremlins else dict(CFG)
    a = make_env(backend, n, names, seed, cfg, robot=robot, max_episode_steps=T)
    b = make_env(backend, n, names, seed, cfg, robot=robot, max_episode_steps=T)
    dev = _dev(a)
    offsets = np.arange(n) % T
    _stagger((a, b), offsets)
    if moving:
        _set_bodies_moving((a, b))
    queued = np.arange(n) % 3 != 2
    new_names = [MIXED[(MIXED.index(names[e]) + 3) % len(MIXED)] if names[e] in MIXED else "push_box" for e in range(n)]
    new_names[0] = names[0]   # the same id again still starts a fresh Task instance
    a.set_next_task([TASKS[new_names[e]]() if queued[e] else None for e in range(n)])
    old_ids = a.task_ids.cpu().numpy().copy()
    want_ids = np.where(queued, [TASK_IDS[x] for x in new_names], old_ids)
    old_f64 = a.get_field("task_f64").cpu().numpy().copy()
    rng = np.random.RandomState(seed)
    switched = np.zeros(n, dtype=bool)
    for t in range(1, 2 * T + 1):
        act = torch.from_numpy(rng.uniform(-1, 1, (n, 2)).astype(np.float32)).to(dev)
        sa, sb = _snap(a.step(act)), _snap(b.step(act))
        np.testing.assert_array_equal(sa[2].cpu().numpy(), sb[2].cpu().numpy(), err_msg=f"done, step {t}")
        np.testing.assert_array_equal(sa[5].cpu().numpy(), sb[5].cpu().numpy(), err_msg=f"truncated, step {t}")
        ends = sa[2].cpu().numpy()   # episodes that ended in this step (time limit, or done): their environments were reset
        keep = ~(queued & (switched | ends))     # rows of environments that run what the twin runs
        for x, y in zip(sa[:5], sb[:5]):
            np.testing.assert_array_equal(x.cpu().numpy()[keep], y.cpu().numpy()[keep], err_msg=f"step {t}")
        ids = a.task_ids.cpu().numpy()
        slot = a.get_field("next_task").cpu().numpy()[:n]
        for e in np.nonzero(queued & ends & ~switched)[0]:
            assert ids[e] == want_ids[e] and slot[e] == -1, (t, e)
            o = _check_fresh_instance(a, e, robot, cfg, seed)
            np.testing.assert_array_equal(sa[0][e].cpu().numpy(), o.observation().astype(np.float32), err_msg=f"first obs of env {e}")
            assert sa[4][e].item() == o.bound
            switched[e] = True
        pending = queued & ~switched
        assert (ids[pending] == old_ids[pending]).all() and (slot[pending] == want_ids[pending]).all(), t
    assert switched[queued].all()
    # fresh instances: new bound draws for the switched environments
    new_f64 = a.get_field("task_f64").cpu().numpy()
    assert (new_f64[14, :n][queued] != old_f64[14, :n][queued]).all()
    assert (a.get_field("next_task").cpu().numpy() == -1).all()
    ra, oa = env_state(a)
    rb, ob = env_state(b)
    np.testing.assert_array_equal(ra[~queued], rb[~queued])
    np.testing.assert_array_equal(oa[~queued], ob[~queued])
    for name in ("task_f64", "task_i32", "flags"):
        np.testing.assert_array_equal(a.get_field(name).cpu().numpy()[..., :n][..., ~queued],
                                      b.get_field(name).cpu().numpy()[..., :n][..., ~queued], err_msg=name)
    a.close(); b.close()


def run_follow_oracle(backend, robot="point", steps_after=50, seed=13):
    """After the switch the environment IS the oracle's fresh Task instance: state at the switch and 50 more steps of
    obs / reward / cost / done, bit for bit, with random_bound and robot_ctrl_range_scale on."""
    n, limit = 6, 60
    names = ["go_to_goal", "push_box", "press_buttons"] * 2
    new = ["push_box", "press_buttons", "go_to_goal", "collect", "go_to_goal", "haul_box"]
    env = make_env(backend, n, names, seed, CFG, robot=robot, max_episode_steps=limit)
    dev = _dev(env)
    _stagger([env], limit - 1 - (np.arange(n) % 3))   # the episodes end at steps 1, 2, 3
    env.set_next_task([TASKS[x]() for x in new])
    rng = np.random.RandomState(seed)
    orc = [None] * n
    for t in range(1, 4 + steps_after):
        act_np = rng.uniform(-1, 1, (n, 2)).astype(np.float32)
        obs, rew, done, info = env.step(torch.from_numpy(act_np).to(dev))
        obs, rew, cost = obs.cpu().numpy(), rew.cpu().numpy(), info["cost"].cpu().numpy()
        done, trunc, bound = done.cpu().numpy(), info["truncated"].cpu().numpy(), info["bound"].cpu().numpy()
        for e in range(n):
            if orc[e] is not None:
                oobs, orew, ocost, odone, rc = orc[e].step(act_np[e].astype(np.float64))
                msg = f"env {e} step {t}"
                assert rc == 0 and cost[e] == ocost and bool(done[e]) == odone and not trunc[e], msg
                assert rew[e] == orew[0], msg
                np.testing.assert_array_equal(obs[e], oobs.astype(np.float32), err_msg=msg)
                assert bound[e] == orc[e].bound, msg
            elif trunc[e]:
                assert t == 1 + e % 3
                orc[e] = _check_fresh_instance(env, e, robot, CFG, seed)
                assert env.task_ids[e].item() == TASK_IDS[new[e]]
                np.testing.assert_array_equal(obs[e], orc[e].observation().astype(np.float32))
    assert all(o is not None for o in orc)
    r, objs = env_state(env)
    ro, oo = oracle_state(orc)
    np.testing.assert_array_equal(r, ro)
    for e, o in enumerate(orc):
        np.testing.assert_array_equal(objs[e, :o.nobj], oo[e, :o.nobj], err_msg=f"objects of env {e}")
    env.close()


def run_stats_follow_task(backend):
    """Finished episodes stay with the task they ran under across switches; a set_task(mask) that cuts an unfinished
    episode does not count it."""
    n = 4
    env = make_env(backend, n, "go_to_goal", 22, {"action_noise": 0.0}, max_episode_steps=T)
    act = torch.zeros((n, 2), device=env.device)
    _stagger([env], [0, 2, 4, 6])
    env.set_next_task(tasks.PushBox())
    gtg, pb = tasks.GoToGoal.task_id, tasks.PushBox.task_id
    for _ in range(T):           # every environment finishes one go_to_goal episode and switches
        env.step(act)
    st = env.task_stats().cpu().numpy()
    assert st[gtg, 2] == n and st[pb, 2] == 0, st[:, 2]
    assert (env.task_ids.cpu().numpy() == pb).all()
    ret_gtg = st[gtg, 0]
    for _ in range(T):           # one push_box episode each
        env.step(act)
    st = env.task_stats().cpu().numpy()
    assert st[gtg, 2] == n and st[pb, 2] == n and st[gtg, 0] == ret_gtg, st[:, 2]
    # cut the running push_box episodes of environments 0 and 2 (0 has just started one, 2 is 4 steps into it): not
    # counted; 1 and 3 run on
    env.set_task(tasks.GoToGoal(), mask=[True, False, True, False])
    np.testing.assert_array_equal(env.task_ids.cpu().numpy(), [gtg, pb, gtg, pb])
    st2 = env.task_stats().cpu().numpy()
    np.testing.assert_array_equal(st2, st)
    env.close()


def run_bad_id_not_applied(backend):
    """A bad id written into the slot with sag_write_field is not applied: the slot is cleared, the environment resets
    as if nothing had been queued and SAG_ERR_BAD_TASK_ID is raised."""
    n = 4
    a = make_env(backend, n, "go_to_goal", 23, {"action_noise": 0.0}, max_episode_steps=T)
    b = make_env(backend, n, "go_to_goal", 23, {"action_noise": 0.0}, max_episode_steps=T)
    slot = a.get_field("next_task")
    slot[1] = 99
    slot[2] = -7
    a.set_field("next_task", slot)
    act = torch.zeros((n, 2), device=a.device)
    for _ in range(T - 1):
        a.step(act); b.step(act)
    a.check_errors()
    with pytest.raises(ValueError, match="task id"):
        a.step(act)
    b.step(act)
    assert (a.get_field("next_task").cpu().numpy() == -1).all()
    for name in a._FIELDS:
        np.testing.assert_array_equal(a.get_field(name).cpu().numpy(), b.get_field(name).cpu().numpy(), err_msg=name)
    a.close(); b.close()


def run_state_dict_resumes(backend, seed=29):
    n = 6
    cfg = dict(CFG)
    a = make_env(backend, n, MIXED[:n], seed, cfg, max_episode_steps=T)
    b = make_env(backend, n, MIXED[:n], seed + 1, cfg, max_episode_steps=T)
    _stagger([a], np.arange(n) % T)
    dev = _dev(a)
    act = torch.zeros((n, 2), device=dev)
    a.step(act)
    a.set_next_task([TASKS[MIXED[(k + 2) % len(MIXED)]]() if k % 2 == 0 else None for k in range(n)])
    sd = a.state_dict()
    assert (sd["fields"]["next_task"][:n].numpy() >= 0).sum() == 3
    b.load_state_dict(sd)
    rng = np.random.RandomState(seed)
    for t in range(2 * T):
        act = torch.from_numpy(rng.uniform(-1, 1, (n, 2)).astype(np.float32)).to(dev)
        for x, y in zip(_snap(a.step(act)), _snap(b.step(act))):
            np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy(), err_msg=f"step {t}")
    for name in a._FIELDS:
        np.testing.assert_array_equal(a.get_field(name).cpu().numpy(), b.get_field(name).cpu().numpy(), err_msg=name)
    # a state_dict saved before tasks could be queued loads with nothing queued
    b.set_next_task(tasks.PushBox())
    old = a.state_dict()
    del old["fields"]["next_task"]
    b.load_state_dict(old)
    assert (b.get_field("next_task").cpu().numpy() == -1).all()
    a.close(); b.close()


# ---- CPU: host-emulated library ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("moving", [False, True])
def test_switch_at_episode_ends_hostemu(moving):
    run_switch_at_episode_ends("hostemu", 9, [MIXED[e % len(MIXED)] for e in range(9)], moving=moving)


def test_switch_follows_oracle_hostemu():
    run_follow_oracle("hostemu")


def test_stats_follow_task_hostemu():
    run_stats_follow_task("hostemu")


def test_bad_id_not_applied_hostemu():
    run_bad_id_not_applied("hostemu")


def test_state_dict_resumes_hostemu():
    run_state_dict_resumes("hostemu")


def test_set_next_task_validates_host_input(monkeypatch):
    env = make_env("hostemu", 4, "go_to_goal", 3)
    with pytest.raises(ValueError, match="need 4"):
        env.set_next_task([tasks.PushBox()] * 3)
    with pytest.raises(ValueError, match="out of range"):
        env.set_next_task(np.array([0, 1, 14, -1]))
    with pytest.raises(ValueError, match="int32"):
        env.set_next_task(torch.zeros(4, dtype=torch.int64))   # a tensor on the env's device must be int32 [N]
    with pytest.raises(ValueError, match="set_task"):
        env.set_next_task([tasks.Unsupervised(), None, None, None])
    monkeypatch.setattr(tasks, "DEVICE_UNSUPPORTED", frozenset({"push_box"}))
    with pytest.raises(NotImplementedError, match="push_box"):
        env.set_next_task([None, tasks.PushBox(), None, None])
    assert (env.get_field("next_task").cpu().numpy() == -1).all()   # nothing was queued by the refused calls
    env.set_next_task(np.array([-1, 3, -1, 8]))
    np.testing.assert_array_equal(env.get_field("next_task").numpy()[:4], [-1, 3, -1, 8])
    # a batch whose reward is already the pair may queue Unsupervised
    u = make_env("hostemu", 2, ["unsupervised", "go_to_goal"], 3)
    u.set_next_task([tasks.GoToGoal(), tasks.Unsupervised()])
    np.testing.assert_array_equal(u.get_field("next_task").numpy()[:2], [3, 13])


def test_whole_batch_set_task_clears_slots():
    env = make_env("hostemu", 4, "go_to_goal", 3)
    env.set_next_task(tasks.PushBox())
    assert (env.get_field("next_task").numpy()[:4] == tasks.PushBox.task_id).all()
    env.set_task(tasks.GoToGoal())
    assert (env.get_field("next_task").numpy() == -1).all()


def test_reset_paths_consume_the_slot():
    """reset_envs(mask) and reset() consume the queued tasks of the environments they reset, and only those."""
    env = make_env("hostemu", 4, "go_to_goal", 5, {"action_noise": 0.0})
    env.set_next_task([tasks.PushBox(), tasks.PushBox(), None, tasks.Collect()])
    env.reset_envs(np.array([True, False, True, False]))
    np.testing.assert_array_equal(env.task_ids.numpy(), [10, 3, 3, 3])
    np.testing.assert_array_equal(env.get_field("next_task").numpy()[:4], [-1, 10, -1, 1])
    env.reset()
    np.testing.assert_array_equal(env.task_ids.numpy(), [10, 10, 3, 1])
    assert (env.get_field("next_task").numpy() == -1).all()


def test_host_input_refused_under_capture(monkeypatch):
    env = make_env("hostemu", 4, "go_to_goal", 3)
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: True)
    with pytest.raises(RuntimeError, match="set_next_task"):
        env.set_next_task(tasks.PushBox())
    with pytest.raises(RuntimeError, match="set_next_task"):
        env.set_next_task([None, tasks.PushBox(), None, None])
    with pytest.raises(RuntimeError, match="set_task"):
        env.set_task(tasks.PushBox(), mask=[True, False, False, False])
    env.set_next_task(torch.tensor([-1, 10, -1, -1], dtype=torch.int32))   # a tensor on the env's device is accepted
    np.testing.assert_array_equal(env.get_field("next_task").numpy()[:4], [-1, 10, -1, -1])


# ---- GPU: the CUDA library --------------------------------------------------------------------------------------------
GPU_CASES = [
    pytest.param("point", 0, "mixed", id="mixed-point"),
    pytest.param("car", 0, "mixed", id="mixed-car"),
    pytest.param("point", 2, "mixed", id="mixed-pointG"),
    pytest.param("car", 2, "push_box", id="push_box-carG"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("robot,gremlins,task", GPU_CASES)
def test_switch_at_episode_ends_cuda(robot, gremlins, task):
    n = 256
    names = [MIXED[e % len(MIXED)] for e in range(n)] if task == "mixed" else [task] * n
    run_switch_at_episode_ends("cuda", n, names, robot=robot, gremlins=gremlins, moving=True)


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["point", "car"])
def test_switch_follows_oracle_cuda(robot):
    run_follow_oracle("cuda", robot=robot)


@pytest.mark.gpu
def test_stats_follow_task_cuda():
    run_stats_follow_task("cuda")


@pytest.mark.gpu
def test_bad_id_not_applied_cuda():
    run_bad_id_not_applied("cuda")


@pytest.mark.gpu
def test_state_dict_resumes_cuda():
    run_state_dict_resumes("cuda")


class _Policy:
    """Fixed-weight two-layer MLP written with broadcast products and sums, so that its arithmetic is the same inside
    and outside a graph."""

    def __init__(self, obs_dim, hidden=16, seed=0):
        g = torch.Generator().manual_seed(seed)
        self.w1 = (torch.randn((obs_dim, hidden), generator=g) / obs_dim ** 0.5).cuda()
        self.w2 = (torch.randn((hidden, 2), generator=g) / hidden ** 0.5).cuda()

    def __call__(self, obs):
        h = torch.tanh((obs[:, :, None] * self.w1[None]).sum(1))
        return torch.tanh((h[:, :, None] * self.w2[None]).sum(1))


def _next_ids(env, schedule, per_task):
    """Device-side schedule walk: an environment whose next episode starts a new block of `per_task` episodes queues
    the next task of its row of `schedule` [N, K]; the others queue nothing."""
    nxt = env.get_field("task_i32")[8, :env.num_envs].to(torch.int64) + 1   # the next episode's number
    k = (nxt // per_task) % schedule.shape[1]
    ids = schedule.gather(1, k[:, None])[:, 0]
    return torch.where(nxt % per_task == 0, ids, torch.full_like(ids, -1))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3])
def test_graphed_adaptation_loop_matches_eager(k):
    """policy + set_next_task(schedule[...]) + step in one CUDA graph, walking a per-environment [N, K] schedule with 3
    episodes per task, over more than 3 K short episodes: bit-identical to an eager twin issuing the same calls."""
    n, K, per_task = 256, 4, 3
    cfg = dict(CFG)
    ge = make_env("cuda", n, MIXED * (n // len(MIXED)), 71, cfg, max_episode_steps=T, copy_outputs=False)
    ee = make_env("cuda", n, MIXED * (n // len(MIXED)), 71, cfg, max_episode_steps=T, copy_outputs=False)
    _stagger((ge, ee), np.arange(n) % T)
    _set_bodies_moving((ge, ee))
    g = torch.Generator().manual_seed(3)
    schedule = torch.randint(0, len(MIXED), (n, K), generator=g)
    schedule = torch.tensor([TASK_IDS[x] for x in MIXED])[schedule].to(torch.int32).cuda()
    schedule[:, 0] = ge.task_ids
    pi = _Policy(ge.obs_dim)
    g_obs, e_obs = ge.observation.clone(), ee.observation.clone()

    def body(env, obs):
        env.set_next_task(_next_ids(env, schedule, per_task))
        out = env.step(pi(obs))
        obs.copy_(out[0])
        return _snap(out)

    a, b = body(ge, g_obs), body(ee, e_obs)   # warm-up: loads every kernel, arms the bound refresh
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        snaps = [body(ge, g_obs) for _ in range(k)]
    seen = set()
    for r in range(-(-((K * per_task + 2) * T) // k)):
        graph.replay()
        for i in range(k):
            want = body(ee, e_obs)
            for x, y in zip(snaps[i], want):
                np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy(), err_msg=f"replay {r} step {i}")
        seen.update(ge.task_ids.cpu().numpy()[:8].tolist())
    for name in ge._FIELDS:
        np.testing.assert_array_equal(ge.get_field(name).cpu().numpy(), ee.get_field(name).cpu().numpy(), err_msg=name)
    ep = ge.get_field("task_i32")[8, :n].cpu().numpy()
    assert ep.min() > per_task * K   # every environment walked its whole schedule and started over
    ids = ge.task_ids.cpu().numpy()
    want = schedule.cpu().numpy()[np.arange(n), (ep // per_task) % K]
    np.testing.assert_array_equal(ids, want)
    assert len(seen) > 2
    ge.check_errors()


@pytest.mark.gpu
def test_fullsize_switches_match_oracle():
    """65,536 point environments with staggered episodes, a task switch at every episode end, 1,100 steps; 256 sampled
    global ids are compared at every switch with oracle environments built for that task and episode, and stepped
    along with them until their next switch."""
    n, limit, steps, seed = 65536, 250, 1100, 666
    cycle = ["go_to_goal", "push_box", "press_buttons", "collect", "go_to_goal_scarce", "catch_goal"]
    cfg = {"action_noise": 0.01, "random_bound": True, "robot_ctrl_range_scale": 0.3}
    env = make_env("cuda", n, [cycle[e % len(cycle)] for e in range(n)], seed, cfg, max_episode_steps=limit, copy_outputs=False)
    rs = np.random.RandomState(seed)
    _stagger([env], rs.randint(0, limit, n))
    ids = np.array(sorted(rs.choice(n, 256, replace=False)))
    idt = torch.as_tensor(ids, device="cuda")
    cyc = torch.tensor([TASK_IDS[x] for x in cycle], dtype=torch.int32, device="cuda")
    pos_of = torch.zeros(_abi.NUM_TASKS, dtype=torch.int64, device="cuda")
    pos_of[cyc.long()] = torch.arange(len(cycle), device="cuda")
    g = torch.Generator(device="cuda").manual_seed(seed)
    orc = [None] * len(ids)
    switches = 0
    for t in range(steps):
        ti = env.get_field("task_i32")[:, :n].to(torch.int64)
        pos = pos_of[ti[0]]   # index of the current task in the cycle; the next one skips a task every other episode
        env.set_next_task(cyc[(pos + 1 + ti[8] % 2) % len(cycle)])
        act = torch.rand((n, 2), device="cuda", generator=g) * 2 - 1
        obs, rew, done, info = env.step(act)
        obs_s, rew_s, cost_s = obs[idt].cpu().numpy(), rew[idt].cpu().numpy(), info["cost"][idt].cpu().numpy()
        done_s, trunc_s, bound_s = done[idt].cpu().numpy(), info["truncated"][idt].cpu().numpy(), info["bound"][idt].cpu().numpy()
        acts = act[idt].cpu().numpy()
        for j, e in enumerate(ids):
            if orc[j] is not None:
                oobs, orew, ocost, odone, rc = orc[j].step(acts[j].astype(np.float64))
                msg = f"global env {e} step {t}"
                assert rc == 0 and float(cost_s[j]) == ocost and float(rew_s[j]) == orew[0], msg
                assert bool(done_s[j]) == (odone or bool(trunc_s[j])), msg
                if not trunc_s[j]:
                    np.testing.assert_array_equal(obs_s[j], oobs.astype(np.float32), err_msg=msg)
            if trunc_s[j]:
                orc[j] = _check_fresh_instance(env, int(e), "point", cfg, seed)
                np.testing.assert_array_equal(obs_s[j], orc[j].observation().astype(np.float32), err_msg=f"env {e} step {t}")
                assert bound_s[j] == orc[j].bound
                switches += 1
    assert switches >= 3 * len(ids)
    env.check_errors()
    env.close()


@pytest.mark.gpu
def test_set_next_tasks_host_through_ctypes():
    """The C entry point as the INTEGRATION.md stub calls it: validated, synchronous, consumed by sag_reset_host."""
    lib = _abi.load()
    L = lib.L
    cfg = lib.default_config()
    cfg.n_envs, cfg.seed = 8, 5
    h = C.c_void_p()
    lib.check(L.sag_create(C.byref(cfg), 0, C.byref(h)))
    try:
        ids = (C.c_int32 * 8)(*([3] * 8))
        lib.check(L.sag_set_tasks_host(h, ids))
        lib.check(L.sag_reset_host(h, None, 0, 1, None))
        bad = (C.c_int32 * 8)(*([-1] * 7 + [14]))
        assert L.sag_set_next_tasks_host(h, bad) != 0 and b"out of range" in L.sag_last_error()
        nxt = (C.c_int32 * 8)(*[10, -1, 8, -1, -1, -1, -1, 1])
        lib.check(L.sag_set_next_tasks_host(h, nxt))
        lib.check(L.sag_reset_host(h, None, 0, 0, None))
        ti = torch.empty((10, 32), dtype=torch.int32, device="cuda")
        lib.check(L.sag_read_field(h, _abi.F_TASK_I32, C.c_void_p(ti.data_ptr()), None))
        slot = torch.empty((32,), dtype=torch.int32, device="cuda")
        lib.check(L.sag_read_field(h, _abi.F_NEXT_TASK, C.c_void_p(slot.data_ptr()), None))
        torch.cuda.synchronize()
        np.testing.assert_array_equal(ti[0, :8].cpu().numpy(), [10, 3, 8, 3, 3, 3, 3, 1])
        assert (slot.cpu().numpy() == -1).all()
        bound = (C.c_double * 8)()
        lib.check(L.sag_bound_host(h, bound))
        bd = torch.empty((8,), dtype=torch.float64, device="cuda")
        lib.check(L.sag_bound(h, C.c_void_p(bd.data_ptr()), None))
        torch.cuda.synchronize()
        np.testing.assert_array_equal(bd.cpu().numpy(), np.array(bound[:]))
        assert L.sag_error_flags(h, 1) == 0
    finally:
        L.sag_destroy(h)
