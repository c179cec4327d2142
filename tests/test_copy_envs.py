"""Environment copies within and across batches (env.copy_envs, sag_copy_envs).  Each case runs on the host emulation
with the copy entry points (CPU, tests/hostemu/sag_hostemu_copy.cpp) and on the CUDA library (-m gpu): a copied
environment's fields must equal its source's bit for bit, a copy with its source's global id must replay the source,
and a copy with another global id must equal an oracle environment of that id injected with the source's state."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import common
import oracle as O
from safe_adaptation_gym_b200 import _abi, tasks
from safe_adaptation_gym_b200.benchmark import TASKS
from safe_adaptation_gym_b200.env import BatchedSafeAdaptationGym

HOSTEMU_SRC = os.path.join(common.ROOT, "tests", "hostemu", "sag_hostemu_copy.cpp")
HOSTEMU_LIB = os.path.join(common.ROOT, "tests", "hostemu", "libsag_hostemu_copy.so")
_hostemu = None


def hostemu_lib():
    """g++ build of the host emulation with the copy entry points (tests/hostemu/sag_hostemu_copy.cpp)."""
    global _hostemu
    if _hostemu is None:
        deps = [HOSTEMU_SRC, common.HOSTEMU_SRC, os.path.join(common.ROOT, "tests", "hostemu", "sag_hostemu_next_task.cpp")] + [
            os.path.join(common.ROOT, p) for p in (
                "safe_adaptation_gym_b200/csrc/sag_core.cuh", "safe_adaptation_gym_b200/csrc/sag_layout.h",
                "include/sag_b200.h", "include/sag_detmath.h")]
        if not os.path.exists(HOSTEMU_LIB) or os.path.getmtime(HOSTEMU_LIB) < max(os.path.getmtime(d) for d in deps):
            fma = ["-mfma"] if "fma" in open("/proc/cpuinfo").read().split() else []
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off"] + fma +
                                  ["-o", HOSTEMU_LIB, HOSTEMU_SRC])
        _hostemu = _abi.SagLib(HOSTEMU_LIB, host_api=False)
    return _hostemu


def make_env(backend, n, task_names, seed, config=None, robot="point", **kw):
    """common.make_env, with the host emulation that has the copy entry points for backend 'hostemu'."""
    if backend != "hostemu":
        return common.make_env(backend, n, task_names, seed, config, robot=robot, **kw)
    env = BatchedSafeAdaptationGym("xmls/%s.xml" % robot, config=config, num_envs=n, _test_lib=hostemu_lib(), **kw)
    env.seed(seed)
    if isinstance(task_names, str):
        task_names = [task_names] * n
    env.set_task([TASKS[t]() for t in task_names])
    return env


MIXED = ["go_to_goal", "press_buttons", "push_box", "collect", "catch_goal", "haul_box", "go_to_goal_scarce", "roll_rod"]
# tasks whose objects keep their lidar groups: an oracle can be injected with their state slot by slot
INJECTABLE = ["go_to_goal", "push_box", "catch_goal", "go_to_goal_scarce"]


def _dev(env):
    return "cuda" if env.device.type == "cuda" else "cpu"


def _fields(env):
    return {name: env.get_field(name).cpu().numpy().copy() for name in env._FIELDS}


def _snap(out):
    obs, rew, done, info = out
    return [t.clone() for t in (obs, rew, done, info["cost"], info["bound"])] + (
        [info["truncated"].clone()] if "truncated" in info else [])


def _steps(envs, k, rng):
    for _ in range(k):
        for env in envs:
            act = torch.from_numpy(rng.uniform(-1, 1, (env.num_envs, 2)).astype(np.float32)).to(_dev(env))
            env.step(act)


def _goal_onto_robot(env, e, task="go_to_goal"):
    """Put the goal of environment e under its robot, so that its next step reaches the goal and resamples it."""
    gremlins = int(env.base_config.get("num_gremlins", 0))
    slot = O.OracleEnv(env.robot_name, task, config={"num_gremlins": gremlins}).slot_types().index(O.GOAL)
    objs, rob = env.get_field("objects"), env.get_field("robot")
    objs[0, slot, e], objs[1, slot, e] = rob[0, e], rob[1, e]
    env.set_field("objects", objs)
    _ = env.observation


def _check_copied(dst, src, idx, before_dst, before_src):
    """every field: dst columns j with idx[j] >= 0 == the source's pre-copy column idx[j]; the others (and the padding)
    unchanged; the source unchanged"""
    n = dst.num_envs
    idx = np.asarray(idx)
    after, after_src = _fields(dst), _fields(src)
    for name in dst._FIELDS:
        want = before_dst[name].copy()
        j = np.nonzero(idx >= 0)[0]
        want[..., j] = before_src[name][..., idx[j]]
        np.testing.assert_array_equal(after[name].view(np.uint8) if after[name].dtype == np.float64 else after[name],
                                      want.view(np.uint8) if want.dtype == np.float64 else want, err_msg=name)
        assert after[name].shape[-1] == dst.stride and n <= dst.stride
        if src is not dst:
            np.testing.assert_array_equal(after_src[name], before_src[name], err_msg="source " + name)


# ---- 1. field identity ------------------------------------------------------------------------------------------------
def run_field_identity(backend, robot="point", gremlins=0, seed=5):
    cfg = {"action_noise": 0.01, "random_bound": True, "robot_ctrl_range_scale": 0.3}
    if gremlins:
        cfg["num_gremlins"] = gremlins
    rng = np.random.RandomState(seed)
    src = make_env(backend, 8, MIXED, seed, cfg, robot=robot, max_episode_steps=6)
    dst = make_env(backend, 12, ["collect"] * 12, seed + 1, cfg, robot=robot, env_id_base=40)
    _steps((src, dst), 4, rng)
    src.set_next_task([tasks.PushBox() if e % 3 == 0 else None for e in range(8)])
    # cross-handle: -1 entries, a broadcast (2 -> 1, 2, 3) and a permutation, as a host list and as a device tensor
    for idx, as_tensor in (([-1, 2, 2, 2, 7, 6, 5, 4, 3, 1, 0, -1], False), ([0, 0, 1, 1, -1, 5, 4, 3, 2, 7, 6, 0], True)):
        b_dst, b_src = _fields(dst), _fields(src)
        obs_src = src.observation.clone()
        dst.copy_envs(torch.tensor(idx, dtype=torch.int32, device=_dev(dst)) if as_tensor else idx, source=src)
        _check_copied(dst, src, idx, b_dst, b_src)
        obs = dst.observation
        j = np.nonzero(np.asarray(idx) >= 0)[0]
        np.testing.assert_array_equal(obs[j].cpu().numpy(), obs_src[np.asarray(idx)[j]].cpu().numpy())
        dst.check_errors()
    # same handle: j <- s only where s keeps its own state
    for idx, as_tensor in (([-1, 0, 0, 3, -1, 4, 4, 7], False), ([5, 5, 2, -1, 5, 5, 6, 6], True)):
        b = _fields(src)
        obs_src = src.observation.clone()
        src.copy_envs(torch.tensor(idx, dtype=torch.int32, device=_dev(src)) if as_tensor else idx)
        _check_copied(src, src, idx, b, b)
        j = np.nonzero(np.asarray(idx) >= 0)[0]
        np.testing.assert_array_equal(src.observation[j].cpu().numpy(), obs_src[np.asarray(idx)[j]].cpu().numpy())
        src.check_errors()
    src.close(); dst.close()


# ---- 2. exact replay --------------------------------------------------------------------------------------------------
def run_exact_replay(backend, robot="point", gremlins=0, seed=7, T=9):
    """Copies whose batch has the source's seed and gives each copy its source's global id replay the source exactly,
    with action noise, goal resamples, auto-resets and a queued task switch; the copied episodes are credited as the
    source credits them."""
    cfg = {"action_noise": 0.01, "random_bound": True}
    if gremlins:
        cfg["num_gremlins"] = gremlins
    names = ["go_to_goal", "catch_goal", "push_box", "press_buttons", "go_to_goal", "collect"]
    src = make_env(backend, 6, names, seed, cfg, robot=robot, max_episode_steps=T, env_id_base=10)
    # global id of destination j is 8 + j: destination j = s + 2 is the copy of source s with its global id
    dst = make_env(backend, 9, "haul_box", seed, cfg, robot=robot, max_episode_steps=T, env_id_base=8)
    rng = np.random.RandomState(seed)
    _steps((src, dst), 3, rng)
    _goal_onto_robot(src, 0)
    _goal_onto_robot(src, 4)
    src.set_next_task([None, tasks.GoToGoal(), None, None, None, None])
    src.task_stats(reset=True)
    dst.task_stats(reset=True)
    idx = np.full(9, -1)
    idx[2:8] = np.arange(6)
    dst.copy_envs(idx, source=src)
    j = idx >= 0
    dev = _dev(src)
    rewards = 0.0
    for t in range(3 * T):
        act_np = rng.uniform(-1, 1, (6, 2)).astype(np.float32)
        act_d = np.zeros((9, 2), np.float32)
        act_d[2:8] = act_np
        a = _snap(src.step(torch.from_numpy(act_np).to(dev)))
        b = _snap(dst.step(torch.from_numpy(act_d).to(dev)))
        for x, y in zip(a, b):
            np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy()[j], err_msg=f"step {t}")
        fa, fb = _fields(src), _fields(dst)
        for name in src._FIELDS:
            np.testing.assert_array_equal(fa[name][..., :6], fb[name][..., 2:8], err_msg=f"{name} step {t}")
        rewards = max(rewards, float(a[1][[0, 4]].max()))
    assert rewards > 0.5   # the goal resamples happened
    assert dst.task_ids[3].item() == tasks.GoToGoal.task_id   # the queued switch came with the copy
    st_src, st_dst = src.task_stats().cpu().numpy(), dst.task_stats().cpu().numpy()
    haul = tasks.HaulBox.task_id   # the task of the destinations 0, 1 and 8, which copied nothing
    assert st_src[haul, 2] == 0 and st_dst[haul, 2] > 0
    st_dst[haul] = 0.0
    np.testing.assert_array_equal(st_dst, st_src)
    assert st_src[:, 2].sum() >= 12
    src.close(); dst.close()


# ---- 3. another global id: the oracle ---------------------------------------------------------------------------------
def inject_oracle(env, e, robot, cfg, seed, gid):
    """An oracle environment with global id `gid` whose state is environment e of `env`, field by field."""
    ti = env.get_field("task_i32")[:, e].cpu().numpy()
    f64 = env.get_field("task_f64")[:, e].cpu().numpy()
    o = O.OracleEnv(robot, int(ti[0]), config=cfg, seed=seed, env_gid=gid)
    assert o.reset(int(ti[8])) == 0            # the episode number (and the slot structure of the task)
    o.robot_state = env.get_field("robot")[:, e].cpu().numpy()
    if robot == "car":
        o.robot_ext = env.get_field("robot_ext")[:, e].cpu().numpy()
    objs = env.get_field("objects")[:, :, e].cpu().numpy()
    for s in range(o.nobj):
        o.set_obj(s, x=objs[0, s], y=objs[1, s], yaw=objs[2, s], vx=objs[3, s], vy=objs[4, s], w=objs[5, s])
    ts = o.task_state
    ts[:13] = [f64[0], f64[1], ti[1], ti[2], ti[3], ti[4], f64[2], f64[3], ti[5], f64[4], f64[5], ti[7], f64[6]]
    ts[14:16] = f64[10:12]
    o.task_state = ts                          # includes the in-step draw counter (ti[7])
    sc = f64[12:14].copy()
    o.L.orc_env_set_ctrlrange(o.h, O._dp(-1.0 * sc), O._dp(sc))
    o.forward()
    return o


def run_oracle_other_id(backend, robot="point", steps=60, seed=13):
    cfg = {"action_noise": 0.01}
    src = make_env(backend, 4, INJECTABLE, seed, cfg, robot=robot)
    dst = make_env(backend, 8, "push_box", seed + 100, cfg, robot=robot, env_id_base=1000)
    rng = np.random.RandomState(seed)
    _steps((src, dst), 5, rng)
    _goal_onto_robot(src, 0)
    idx = [0, 1, 2, 3, 0, -1, 3, 1]
    dst.copy_envs(idx, source=src)
    sel = [e for e in range(8) if idx[e] >= 0]
    orc = {e: inject_oracle(src, idx[e], robot, cfg, seed + 100, 1000 + e) for e in sel}
    dev = _dev(dst)
    goals = 0
    for t in range(steps):
        act = np.zeros((8, 2), np.float32)
        for e in sel:
            act[e] = common.drive_action(orc[e], rng).astype(np.float32)
        obs, rew, done, info = dst.step(torch.from_numpy(act).to(dev))
        obs, rew, cost, done = obs.cpu().numpy(), rew.cpu().numpy(), info["cost"].cpu().numpy(), done.cpu().numpy()
        for e in sel:
            oobs, orew, ocost, odone, rc = orc[e].step(act[e].astype(np.float64))
            msg = f"env {e} step {t}"
            assert rc == 0 and rew[e] == orew[0] and cost[e] == ocost and bool(done[e]) == odone, msg
            np.testing.assert_array_equal(obs[e], oobs.astype(np.float32), err_msg=msg)
            goals += int(orew[0] > 0.5)
    assert goals >= 1
    r, objs = common.env_state(dst)
    ro, oo = common.oracle_state([orc[e] for e in sel])
    np.testing.assert_array_equal(r[sel], ro)
    for k, e in enumerate(sel):
        np.testing.assert_array_equal(objs[e, :orc[e].nobj], oo[k, :orc[e].nobj], err_msg=f"objects of env {e}")
    src.close(); dst.close()


# ---- 4. statistics ----------------------------------------------------------------------------------------------------
def run_stats(backend, seed=22, T=5):
    gtg, pb = tasks.GoToGoal.task_id, tasks.PushBox.task_id
    cfg = {"action_noise": 0.0}
    dst = make_env(backend, 4, "go_to_goal", seed, cfg, max_episode_steps=T)
    src = make_env(backend, 2, "push_box", seed, cfg, max_episode_steps=T)
    act4 = torch.zeros((4, 2), device=_dev(dst))
    act2 = torch.full((2, 2), 0.5, device=_dev(src))
    for _ in range(2 * T + 2):    # two finished go_to_goal episodes each, 2 steps into the third
        dst.step(act4)
    for _ in range(3):            # 3 steps into the first push_box episode
        src.step(act2)
    before = dst.task_stats().cpu().numpy()
    assert before[gtg, 2] == 8
    dst.copy_envs([0, 1, -1, -1], source=src)
    st = dst.task_stats().cpu().numpy()
    np.testing.assert_array_equal(st, before)   # the earlier episodes stay with go_to_goal; nothing else counted
    act4[:2] = 0.5
    for _ in range(2):            # the copies finish their push_box episode; 2 and 3 are 4 steps into theirs
        dst.step(act4)
        src.step(act2)
    st = dst.task_stats().cpu().numpy()
    np.testing.assert_array_equal(st[gtg], before[gtg])
    np.testing.assert_array_equal(st[pb], src.task_stats().cpu().numpy()[pb])   # credited in full, as the source does
    assert st[pb, 2] == 2
    dst.close(); src.close()


# ---- 5. rules ---------------------------------------------------------------------------------------------------------
def run_bad_pairs_device(backend):
    env = make_env(backend, 6, "go_to_goal", 3, {"action_noise": 0.0})
    env.step(torch.zeros((6, 2), device=_dev(env)))
    b = _fields(env)
    # 0 <- 1 (1 is overwritten), 1 <- 2 (fine), 3 <- 9 and 4 <- -5 (out of range), 5 <- 5 (nothing)
    env.copy_envs(torch.tensor([1, 2, -1, 9, -5, 5], dtype=torch.int32, device=_dev(env)))
    _check_copied(env, env, [-1, 2, -1, -1, -1, -1], b, b)
    with pytest.raises(IndexError, match="copy_envs"):
        env.check_errors()
    env.check_errors()   # cleared
    env.close()


def run_stats_ended_not_reset(backend):
    """A destination whose episode has finished but has not been reset yet: the copy counts that episode under the old
    task, as reset_envs does, before the destination takes the copied state."""
    gtg, pb = tasks.GoToGoal.task_id, tasks.PushBox.task_id
    cfg = {"action_noise": 0.0}
    a, b = (make_env(backend, 3, "go_to_goal", 22, cfg) for _ in range(2))
    src = make_env(backend, 2, "push_box", 23, cfg)
    act = torch.full((3, 2), 0.3, device=_dev(a))
    for _ in range(3):
        a.step(act)
        b.step(act)
    for env in (a, b):   # environment 0's episode has ended (done or time limit) and waits for its reset
        fl = env.get_field("flags")
        fl[0] |= _abi.FLAG_NEEDS_RESET
        env.set_field("flags", fl)
    a.copy_envs([1, -1, -1], source=src)
    b.reset_envs(np.array([True, False, False]))
    sa, sb = a.task_stats().cpu().numpy(), b.task_stats().cpu().numpy()
    assert sa[gtg, 2] == 1 and sa[pb, 2] == 0, sa[:, 2]
    np.testing.assert_array_equal(sa, sb)
    for env in (a, b, src):
        env.close()


def run_host_input_is_validated(backend):
    env = make_env(backend, 4, "go_to_goal", 3)
    other = make_env(backend, 3, "push_box", 4)
    b = _fields(env)
    with pytest.raises(ValueError, match="need 4"):
        env.copy_envs([0, 1, 2])
    with pytest.raises(ValueError, match="integers"):
        env.copy_envs(np.array([0.0, 1.0, -1.0, -1.0]))
    with pytest.raises(ValueError, match="int32"):   # a tensor on the env's device must be int32 [N]
        env.copy_envs(torch.zeros(4, dtype=torch.int64, device=_dev(env)))
    with pytest.raises(IndexError, match="out of range"):
        env.copy_envs([0, 3, -1, 4])
    with pytest.raises(IndexError, match="out of range"):
        env.copy_envs([-1, -1, 3, -1], source=other)
    with pytest.raises(IndexError, match="out of range"):
        env.copy_envs([-2, -1, -1, -1])
    with pytest.raises(ValueError, match="overwrites"):
        env.copy_envs([1, 2, -1, -1])
    _check_copied(env, env, [-1] * 4, b, b)   # nothing was copied by the refused calls
    env.copy_envs(np.array([-1, 0, 1, 2], dtype=np.int16), source=other)
    env.check_errors()
    # the C entry point validates as well
    L = env._lib
    bad = (C.c_int32 * 4)(1, 2, -1, -1)
    assert L.L.sag_copy_envs_host(env._h, env._h, bad) != 0 and b"overwritten" in L.L.sag_last_error()
    bad = (C.c_int32 * 4)(-1, 3, -1, -1)
    assert L.L.sag_copy_envs_host(env._h, other._h, bad) != 0 and b"out of range" in L.L.sag_last_error()
    env.close(); other.close()


def run_incompatible_batches_are_refused(backend):
    base = make_env(backend, 4, "go_to_goal", 3)
    idx = [0, 1, -1, -1]
    L = base._lib
    arr = (C.c_int32 * 4)(*idx)
    dev_arr = torch.tensor(idx, dtype=torch.int32, device=_dev(base))
    for kw in ({"robot": "car"}, {"config": {"num_gremlins": 1}}, {"config": {"hazards_size": 0.25}},
               {"config": {"pillars_keepout": 0.5}}, {"config": {"random_bound": True}}, {"config": {"max_bound": 10}},
               {"config": {"robot_ctrl_range_scale": 0.1}}, {"config": {"placements_margin": 0.1}}):
        other = make_env(backend, 4, "go_to_goal", 3, **kw)
        with pytest.raises(ValueError, match="differ"):
            base.copy_envs(idx, source=other)
        with pytest.raises(ValueError, match="differ"):
            other.copy_envs(dev_arr, source=base)
        # the library refuses the pair too, on both paths, and enqueues nothing
        assert L.L.sag_copy_envs_host(base._h, other._h, arr) != 0 and b"differ" in L.L.sag_last_error()
        assert L.L.sag_copy_envs(other._h, base._h, C.c_void_p(dev_arr.data_ptr()), base._stream()) != 0
        assert b"differ" in L.L.sag_last_error()
        other.close()
    # budgets, seed, global ids and noise may differ, and so may keepouts that the object size overrides
    # (effective keepout = max(keepout, size), world.py:60-66: 0.15 and 0.1 against a hazard size of 0.2)
    plan = make_env(backend, 6, "push_box", 9, {"action_noise": 0.0, "hazards_keepout": 0.1}, max_episode_steps=3,
                    env_id_base=77)
    keep = make_env(backend, 4, "go_to_goal", 3, {"hazards_keepout": 0.15})
    plan.copy_envs([0, 1, 2, 3, 3, -1], source=base)
    plan.copy_envs([-1, -1, -1, -1, -1, 0], source=keep)
    np.testing.assert_array_equal(plan.task_ids.cpu().numpy(), [3] * 6)
    plan.check_errors()
    for env in (base, plan, keep):
        env.close()


def run_host_input_refused_under_capture(backend, monkeypatch):
    env = make_env(backend, 4, "go_to_goal", 3)
    idx = torch.tensor([-1, 0, -1, -1], dtype=torch.int32, device=_dev(env))
    if backend == "hostemu":
        monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: True)
        with pytest.raises(RuntimeError, match="copy_envs"):
            env.copy_envs([-1, 0, -1, -1])
        env.copy_envs(idx)   # a tensor on the env's device is accepted
        monkeypatch.undo()
    else:
        with pytest.raises(RuntimeError, match="copy_envs"):
            with torch.cuda.graph(torch.cuda.CUDAGraph()):
                env.copy_envs([-1, 0, -1, -1])
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):   # a tensor on the env's device is recorded
            env.copy_envs(idx)
        rob = env.get_field("robot")
        assert not torch.equal(rob[:, 1], rob[:, 0])   # recorded, not run
        g.replay()
    rob = env.get_field("robot")
    np.testing.assert_array_equal(rob[:, 1].cpu().numpy(), rob[:, 0].cpu().numpy())
    env.check_errors()
    env.close()


def run_unsupervised_rule(backend):
    src = make_env(backend, 2, ["go_to_goal", "unsupervised"], 3)
    dst = make_env(backend, 2, "go_to_goal", 4)
    dst.copy_envs([0, -1], source=src)   # go_to_goal only: fine
    with pytest.raises(ValueError, match="Unsupervised"):
        dst.copy_envs([1, -1], source=src)
    with pytest.raises(ValueError, match="Unsupervised"):   # a device tensor: refused whenever the source has the pair
        dst.copy_envs(torch.tensor([0, -1], dtype=torch.int32, device=_dev(dst)), source=src)
    src2 = make_env(backend, 2, "go_to_goal", 3)
    nt = src2.get_field("next_task")
    nt[1] = tasks.Unsupervised.task_id   # queued (written as a field, as a device-side schedule could)
    src2.set_field("next_task", nt)
    with pytest.raises(ValueError, match="Unsupervised"):
        dst.copy_envs([-1, 1], source=src2)
    pair = make_env(backend, 2, ["unsupervised", "go_to_goal"], 5)
    pair.copy_envs([1, 0], source=src)
    np.testing.assert_array_equal(pair.task_ids.cpu().numpy(), [13, 3])
    out = pair.step(torch.zeros((2, 2), device=_dev(pair)))
    assert tuple(out[1].shape) == (2, 2)
    for env in (src, dst, src2, pair):
        env.close()


def run_random_bound_follows(backend):
    cfg = {"random_bound": True, "action_noise": 0.0}
    src = make_env(backend, 4, "go_to_goal", 3, cfg)
    dst = make_env(backend, 4, "go_to_goal", 4, cfg, copy_outputs=False)
    out = dst.step(torch.zeros((4, 2), device=_dev(dst)))
    bound = out[3]["bound"]            # the internal buffer: refreshed in place
    dst.copy_envs([3, -1, 0, 0], source=src)
    sb = src.get_field("task_f64")[14, :4].cpu().numpy()
    want = dst.get_field("task_f64")[14, :4].cpu().numpy()
    np.testing.assert_array_equal(want[[0, 2, 3]], sb[[3, 0, 0]])
    np.testing.assert_array_equal(bound.cpu().numpy(), want)
    out = dst.step(torch.zeros((4, 2), device=_dev(dst)))
    np.testing.assert_array_equal(out[3]["bound"].cpu().numpy(), want)
    src.close(); dst.close()


# ---- CPU: host-emulated library ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("robot,gremlins", [("point", 0), ("car", 0), ("point", 2)])
def test_field_identity_hostemu(robot, gremlins):
    run_field_identity("hostemu", robot, gremlins)


def test_exact_replay_hostemu():
    run_exact_replay("hostemu")


@pytest.mark.parametrize("robot", ["point", "car"])
def test_oracle_other_id_hostemu(robot):
    run_oracle_other_id("hostemu", robot)


def test_stats_hostemu():
    run_stats("hostemu")


def test_stats_ended_not_reset_hostemu():
    run_stats_ended_not_reset("hostemu")


def test_copy_rules_hostemu():
    run_bad_pairs_device("hostemu")


def test_host_input_is_validated_hostemu():
    run_host_input_is_validated("hostemu")


def test_incompatible_batches_are_refused_hostemu():
    run_incompatible_batches_are_refused("hostemu")


def test_host_input_refused_under_capture_hostemu(monkeypatch):
    run_host_input_refused_under_capture("hostemu", monkeypatch)


def test_unsupervised_rule_hostemu():
    run_unsupervised_rule("hostemu")


def test_random_bound_follows_hostemu():
    run_random_bound_follows("hostemu")


# ---- GPU: the CUDA library --------------------------------------------------------------------------------------------
GPU_BUILDS = [pytest.param("point", 0, id="point"), pytest.param("car", 0, id="car"),
              pytest.param("point", 2, id="pointG"), pytest.param("car", 2, id="carG")]


@pytest.mark.gpu
@pytest.mark.parametrize("robot,gremlins", GPU_BUILDS)
def test_field_identity_cuda(robot, gremlins):
    run_field_identity("cuda", robot, gremlins)


@pytest.mark.gpu
@pytest.mark.parametrize("robot,gremlins", GPU_BUILDS)
def test_exact_replay_cuda(robot, gremlins):
    run_exact_replay("cuda", robot, gremlins)


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["point", "car"])
def test_oracle_other_id_cuda(robot):
    run_oracle_other_id("cuda", robot)


@pytest.mark.gpu
def test_stats_cuda():
    run_stats("cuda")


@pytest.mark.gpu
def test_stats_ended_not_reset_cuda():
    run_stats_ended_not_reset("cuda")


@pytest.mark.gpu
def test_copy_rules_cuda():
    run_bad_pairs_device("cuda")


@pytest.mark.gpu
def test_host_input_is_validated_cuda():
    run_host_input_is_validated("cuda")


@pytest.mark.gpu
def test_incompatible_batches_are_refused_cuda():
    run_incompatible_batches_are_refused("cuda")


@pytest.mark.gpu
def test_host_input_refused_under_capture_cuda(monkeypatch):
    run_host_input_refused_under_capture("cuda", monkeypatch)


@pytest.mark.gpu
def test_unsupervised_rule_cuda():
    run_unsupervised_rule("cuda")


@pytest.mark.gpu
def test_device_spellings_and_other_devices():
    """'cuda' and 'cuda:0' name the same device; a batch on another device is refused by Python and by the library."""
    a = make_env("cuda", 4, "go_to_goal", 3, device="cuda")
    b = make_env("cuda", 4, "go_to_goal", 4, device="cuda:0")
    b.copy_envs([1, -1, -1, -1], source=a)
    np.testing.assert_array_equal(b.get_field("robot")[:, 0].cpu().numpy(), a.get_field("robot")[:, 1].cpu().numpy())
    if torch.cuda.device_count() > 1:
        c = make_env("cuda", 4, "go_to_goal", 5, device="cuda:1")
        with pytest.raises(ValueError, match="device"):
            b.copy_envs([1, -1, -1, -1], source=c)
        L = b._lib
        assert L.L.sag_copy_envs_host(b._h, c._h, (C.c_int32 * 4)(1, -1, -1, -1)) != 0
        assert b"different devices" in L.L.sag_last_error()
        c.close()
    a.close(); b.close()


@pytest.mark.gpu
def test_random_bound_follows_cuda():
    run_random_bound_follows("cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("H", [1, 4])
def test_graphed_lookahead_matches_eager(H):
    """copy_envs (K copies of every environment of the main batch) + H candidate steps, accumulating return and cost,
    in one CUDA graph: bit-identical to an eager planning batch issuing the same calls, over several rounds with the
    main batch stepping in between."""
    N, K, seed = 32, 8, 31
    env = make_env("cuda", N, MIXED * (N // len(MIXED)), seed, {"action_noise": 0.01}, max_episode_steps=20)
    plans = [make_env("cuda", N * K, "go_to_goal", seed + 1, {"action_noise": 0.0}, copy_outputs=False) for _ in range(2)]
    src_of = torch.arange(N * K, device="cuda", dtype=torch.int32) // K
    cand = torch.zeros((H, N * K, 2), device="cuda")
    acc = [torch.zeros((2, N * K), dtype=torch.float64, device="cuda") for _ in range(2)]

    def lookahead(plan, ret):
        plan.copy_envs(src_of, source=env)
        ret.zero_()
        for h in range(H):
            _, rew, _, info = plan.step(cand[h])
            ret[0] += rew
            ret[1] += info["cost"]

    g = torch.Generator(device="cuda").manual_seed(seed)
    lookahead(plans[0], acc[0])   # warm-up
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        lookahead(plans[0], acc[0])
    for r in range(6):
        cand.copy_(torch.rand((H, N * K, 2), device="cuda", generator=g) * 2 - 1)
        graph.replay()
        lookahead(plans[1], acc[1])
        np.testing.assert_array_equal(acc[0].cpu().numpy(), acc[1].cpu().numpy(), err_msg=f"round {r}")
        for name in plans[0]._FIELDS:
            np.testing.assert_array_equal(plans[0].get_field(name).cpu().numpy(), plans[1].get_field(name).cpu().numpy(),
                                          err_msg=f"{name} round {r}")
        best = (acc[0][0] - acc[0][1]).view(N, K).argmax(1)
        env.step(cand[0].view(N, K, 2)[torch.arange(N, device="cuda"), best])
    assert float(acc[0][1].abs().sum() + acc[0][0].abs().sum()) > 0.0
    env.check_errors()
    for p in plans:
        p.check_errors()


@pytest.mark.gpu
def test_fullsize_broadcast_matches_oracle():
    """1,024 sources x 64 copies = 65,536 environments of another seed and other global ids; 256 sampled copies are
    stepped along with oracle environments injected with their source's state, bit for bit."""
    n_src, K, seed, steps = 1024, 64, 666, 30
    cfg = {"action_noise": 0.01}
    env = make_env("cuda", n_src, [INJECTABLE[e % len(INJECTABLE)] for e in range(n_src)], seed, cfg)
    plan = make_env("cuda", n_src * K, "go_to_goal", seed + 1, cfg, env_id_base=5000, copy_outputs=False)
    g = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(10):
        env.step(torch.rand((n_src, 2), device="cuda", generator=g) * 2 - 1)
    plan.copy_envs(torch.arange(n_src * K, device="cuda", dtype=torch.int32) // K, source=env)
    ids = np.array(sorted(np.random.RandomState(seed).choice(n_src * K, 256, replace=False)))
    orc = [inject_oracle(env, int(e) // K, "point", cfg, seed + 1, 5000 + int(e)) for e in ids]
    idt = torch.as_tensor(ids, device="cuda")
    for t in range(steps):
        act = torch.rand((n_src * K, 2), device="cuda", generator=g) * 2 - 1
        obs, rew, done, info = plan.step(act)
        obs_s, rew_s, cost_s, done_s = obs[idt].cpu().numpy(), rew[idt].cpu().numpy(), info["cost"][idt].cpu().numpy(), done[idt].cpu().numpy()
        acts = act[idt].cpu().numpy()
        for k, o in enumerate(orc):
            oobs, orew, ocost, odone, rc = o.step(acts[k].astype(np.float64))
            msg = f"copy {ids[k]} step {t}"
            assert rc == 0 and float(rew_s[k]) == orew[0] and float(cost_s[k]) == ocost and bool(done_s[k]) == odone, msg
            np.testing.assert_array_equal(obs_s[k], oobs.astype(np.float32), err_msg=msg)
    r, objs = common.env_state(plan)
    ro, oo = common.oracle_state(orc)
    np.testing.assert_array_equal(r[ids], ro)
    plan.check_errors()


@pytest.mark.gpu
def test_copy_envs_host_through_ctypes():
    """The C entry point as the INTEGRATION.md stub calls it: validated, synchronous, every field copied."""
    lib = _abi.load()
    L = lib.L
    hs = []
    try:
        for n, seed in ((4, 5), (6, 9)):
            cfg = lib.default_config()
            cfg.n_envs, cfg.seed = n, seed
            h = C.c_void_p()
            lib.check(L.sag_create(C.byref(cfg), 0, C.byref(h)))
            hs.append(h)
            lib.check(L.sag_set_tasks_host(h, (C.c_int32 * n)(*([3] * n))))
            lib.check(L.sag_reset_host(h, None, 0, 1, None))
        src, dst = hs

        def field(h, f):
            t = torch.empty((L.sag_field_bytes(h, f),), dtype=torch.uint8, device="cuda")
            lib.check(L.sag_read_field(h, f, C.c_void_p(t.data_ptr()), None))
            torch.cuda.synchronize()
            return t.cpu().numpy()
        before = [field(src, f) for f in range(8)]
        bad = (C.c_int32 * 6)(0, 1, 4, -1, -1, -1)
        assert L.sag_copy_envs_host(dst, src, bad) != 0 and b"out of range" in L.sag_last_error()
        idx = (C.c_int32 * 6)(3, 3, -1, 0, 1, 2)
        lib.check(L.sag_copy_envs_host(dst, src, idx))
        ti = torch.empty((10, 32), dtype=torch.int32, device="cuda")
        lib.check(L.sag_read_field(dst, _abi.F_TASK_I32, C.c_void_p(ti.data_ptr()), None))
        ro = torch.empty((6, 32), dtype=torch.float64, device="cuda")
        lib.check(L.sag_read_field(dst, _abi.F_ROBOT, C.c_void_p(ro.data_ptr()), None))
        rs = torch.empty((6, 32), dtype=torch.float64, device="cuda")
        lib.check(L.sag_read_field(src, _abi.F_ROBOT, C.c_void_p(rs.data_ptr()), None))
        torch.cuda.synchronize()
        np.testing.assert_array_equal(ro[:, [0, 1, 3, 4, 5]].cpu().numpy(), rs[:, [3, 3, 0, 1, 2]].cpu().numpy())
        assert (ti[8, :6].cpu().numpy() == 0).all()
        assert all((field(src, f) == b).all() for f, b in enumerate(before))
        assert L.sag_error_flags(dst, 1) == 0
    finally:
        for h in hs:
            L.sag_destroy(h)
