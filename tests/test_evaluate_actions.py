"""Scoring candidate action sequences (env.evaluate_actions, sag_evaluate_actions).  Every case compares a batch that
calls evaluate_actions with an eager twin -- same seed, tasks and state -- that runs H step calls and accumulates the
return and cost with the same weights and masking in torch: the outputs and every state field must agree bit for bit.
The small cases run on the host emulation with the evaluate entry point (CPU, tests/hostemu/sag_hostemu_evaluate.cpp,
which runs the observation-free step instantiations of sag_core.cuh) and on the CUDA library (-m gpu)."""
import os
import subprocess

import numpy as np
import pytest
import torch

import common
import oracle as O
from safe_adaptation_gym_b200 import _abi
from safe_adaptation_gym_b200.benchmark import TASKS
from safe_adaptation_gym_b200.env import BatchedSafeAdaptationGym

HOSTEMU_SRC = os.path.join(common.ROOT, "tests", "hostemu", "sag_hostemu_evaluate.cpp")
HOSTEMU_LIB = os.path.join(common.ROOT, "tests", "hostemu", "libsag_hostemu_evaluate.so")
_hostemu = None

MIXED = ["go_to_goal", "press_buttons", "push_box", "haul_box", "roll_rod", "catch_goal", "collect"]


def hostemu_lib():
    """g++ build of the host emulation with the evaluate entry point (tests/hostemu/sag_hostemu_evaluate.cpp)."""
    global _hostemu
    if _hostemu is None:
        deps = [HOSTEMU_SRC] + [os.path.join(common.ROOT, "tests", "hostemu", f) for f in (
            "sag_hostemu.cpp", "sag_hostemu_next_task.cpp", "sag_hostemu_copy.cpp")] + [
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
    if backend != "hostemu":
        return common.make_env(backend, n, task_names, seed, config, robot=robot, **kw)
    env = BatchedSafeAdaptationGym("xmls/%s.xml" % robot, config=config, num_envs=n, _test_lib=hostemu_lib(), **kw)
    env.seed(seed)
    if isinstance(task_names, str):
        task_names = [task_names] * n
    env.set_task([TASKS[t]() for t in task_names])
    return env


def _dev(env):
    return "cuda" if env.device.type == "cuda" else "cpu"


def _bits(t):
    a = t.cpu().numpy()
    return a.view(np.uint8) if a.dtype == np.float64 or a.dtype == np.float32 else a


def assert_same_bits(a, b, msg=""):
    assert tuple(a.shape) == tuple(b.shape) and a.dtype == b.dtype, (msg, a.shape, b.shape, a.dtype, b.dtype)
    np.testing.assert_array_equal(_bits(a), _bits(b), err_msg=msg)


def assert_same_state(a, b, msg=""):
    for name in a._FIELDS:
        assert_same_bits(a.get_field(name), b.get_field(name), f"{msg} field {name}")
    assert_same_bits(a.task_stats(), b.task_stats(), f"{msg} task_stats")


def twin_evaluate(env, actions, discount):
    """What evaluate_actions computes, from H step calls: ret / cost summed in step order from zero with the products
    w_h * r_h rounded first, up to and including each environment's first done."""
    H, n = actions.shape[0], env.num_envs
    counting = torch.ones((n,), dtype=torch.bool, device=env.device)
    length = torch.zeros((n,), dtype=torch.int32, device=env.device)
    cost = torch.zeros((n,), dtype=torch.float64, device=env.device)
    ret, w, obs = None, 1.0, None
    for h in range(H):
        obs, r, done, info = env.step(actions[h])
        obs, r = obs.clone(), r.clone()
        if ret is None:
            ret = torch.zeros_like(r)
        m = counting.view(-1, *([1] * (r.dim() - 1)))
        ret = torch.where(m, ret + w * r, ret)
        cost = torch.where(counting, cost + w * info["cost"].to(torch.float64), cost)
        length = torch.where(counting, torch.full_like(length, h + 1), length)
        counting = counting & ~done
        w = w * discount
    return obs, ret, cost, length


def twins(backend, n, task_names, seed, cfg, robot="point", warm=0, **kw):
    """Two batches with the same seed and tasks in the same state; with warm > 0 both take the state a live batch
    reached after `warm` random steps (copy_envs), so that late-episode states -- moving bodies, contacts -- are in."""
    a = make_env(backend, n, task_names, seed, cfg, robot=robot, **kw)
    b = make_env(backend, n, task_names, seed, cfg, robot=robot, **kw)
    if warm:
        live = make_env(backend, n, task_names, seed + 100, cfg, robot=robot)
        rng = np.random.RandomState(seed)
        for _ in range(warm):
            live.step(torch.from_numpy(rng.uniform(-1, 1, (n, 2)).astype(np.float32)).to(_dev(live)))
        idx = torch.arange(n, dtype=torch.int32, device=_dev(live))
        a.copy_envs(idx, source=live)
        b.copy_envs(idx, source=live)
        live.close()
    return a, b


def check_against_twin(a, b, actions, discount, msg=""):
    out = a.evaluate_actions(actions, discount)
    want = twin_evaluate(b, actions, discount)
    for name, x, y in zip(("obs", "ret", "cost", "length"), out, want):
        assert_same_bits(x, y, f"{msg} {name}")
    assert_same_state(a, b, msg)
    a.check_errors()
    b.check_errors()
    return out


def _actions(env, H, seed):
    g = np.random.RandomState(seed)
    return torch.from_numpy(g.uniform(-1, 1, (H, env.num_envs, 2)).astype(np.float32)).to(_dev(env))


# ---- cases --------------------------------------------------------------------------------------------------------
def run_matches_twin(backend, robot, gremlins, tasks, H, discount, n, warm, seed=11):
    cfg = {"action_noise": 0.01}
    if gremlins:
        cfg["num_gremlins"] = gremlins
    names = [MIXED[e % len(MIXED)] for e in range(n)] if tasks == "mixed" else [tasks] * n
    a, b = twins(backend, n, names, seed, cfg, robot=robot, warm=warm)
    for k in range(2):   # two horizons in a row: the second starts where the first left both batches
        obs, ret, cost, length = check_against_twin(a, b, _actions(a, H, seed + k), discount, f"horizon {k}")
        assert tuple(ret.shape) == ((n, 2) if tasks == "unsupervised" else (n,))
        assert bool(((length >= 1) & (length <= H)).all())   # < H after a physics error (contact capacity)
    a.close(); b.close()


def run_physics_error_stops_the_sums(backend, robot, H=8):
    """The capacity overflow of tests/common.py (all vases stacked into one heap the robot drives into): the
    environments' physics error ends their count partway through the horizon; the state still matches the twin."""
    n, cfg = 4, {"action_noise": 0.0}
    a, b = twins(backend, n, "go_to_goal", 77, cfg, robot=robot)
    for env in (a, b):
        objs, rob = env.get_field("objects"), env.get_field("robot")
        for e in range(n):
            rx, ry = float(rob[0, e]), float(rob[1, e])
            for k, s in enumerate(range(9, 19)):          # vase slots
                objs[0, s, e] = rx + 0.16 + 0.03 * (k % 4) + 0.01 * e
                objs[1, s, e] = ry + 0.03 * (k // 4) - 0.03
                objs[2, s, e] = 0.1 * k
            rob[2, e], rob[3, e] = 0.0, 0.5
        env.set_field("objects", objs); env.set_field("robot", rob)
        _ = env.observation
    act = torch.full((H, n, 2), 0.02 if robot == "car" else 0.0, device=_dev(a))
    if robot == "point":
        act[..., 0] = 1.0
    obs, ret, cost, length = check_against_twin(a, b, act, 0.99)
    assert bool((length < H).any()), length
    a.close(); b.close()


def run_goal_resample_inside_horizon(backend, H=5):
    """Goals put under the robots, so that the first step reaches and resamples them: GoToGoal's goal directly, and
    CatchGoal's circle centred on the robot with radius 0 (catch_goal.py:20-31 moves the goal before the reward)."""
    n = 6
    names = ["go_to_goal", "catch_goal"] * 3
    a, b = twins(backend, n, names, 23, {"action_noise": 0.01})
    slot = O.OracleEnv("point", "go_to_goal").slot_types().index(O.GOAL)
    for env in (a, b):
        objs, rob = env.get_field("objects"), env.get_field("robot")
        f64, i32 = env.get_field("task_f64"), env.get_field("task_i32")
        for e in range(0, n, 2):
            objs[0, slot, e], objs[1, slot, e] = rob[0, e], rob[1, e]
        for e in range(1, n, 2):
            f64[2, e] = f64[3, e] = 0.0                       # radius 0
            f64[4, e], f64[5, e] = rob[0, e], rob[1, e]       # circle centre
            i32[5, e] = 5                                     # no radius redraw within the horizon
        env.set_field("objects", objs); env.set_field("task_f64", f64); env.set_field("task_i32", i32)
        _ = env.observation
    goal0 = a.get_field("objects")[:2, slot, 0:n:2].clone()
    _, ret, _, _ = check_against_twin(a, b, torch.zeros((H, n, 2), device=_dev(a)), 0.9)
    assert bool((a.get_field("objects")[:2, slot, 0:n:2] != goal0).any(0).all())   # GoToGoal: resampled
    assert bool((ret > 0.5).all()), ret                                          # the +1 of every reached goal
    a.close(); b.close()


def run_outputs_follow_copy_outputs(backend):
    n, H = 4, 3
    for copy in (True, False):
        env = make_env(backend, n, "go_to_goal", 3, copy_outputs=copy)
        act = torch.zeros((H, n, 2), device=_dev(env))
        first = env.evaluate_actions(act)
        second = env.evaluate_actions(act)
        for x, y in zip(first, second):
            assert (x.data_ptr() == y.data_ptr()) == (not copy)
        assert first[0].dtype == torch.float32 and tuple(first[0].shape) == (n, env.obs_dim)
        assert first[1].dtype == torch.float64 and first[2].dtype == torch.float64 and first[3].dtype == torch.int32
        env.close()


def run_refusals(backend, monkeypatch):
    n = 4
    env = make_env(backend, n, "go_to_goal", 3)
    dev = _dev(env)
    for bad in (torch.zeros((2, n, 2), dtype=torch.float64, device=dev), torch.zeros((2, n, 3), device=dev),
                torch.zeros((n, 2), device=dev), torch.zeros((2, n + 1, 2), device=dev), torch.zeros((0, n, 2), device=dev),
                torch.zeros((2, n, 2), device="meta"), np.zeros((2, n, 2), dtype=np.float32)):
        with pytest.raises(ValueError):
            env.evaluate_actions(bad)
    limited = make_env(backend, n, "go_to_goal", 3, max_episode_steps=10)
    with pytest.raises(ValueError, match="max_episode_steps"):
        limited.evaluate_actions(torch.zeros((2, n, 2), device=dev))
    act = torch.zeros((2, n, 2), device=dev)
    if backend == "hostemu":
        monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: True)
        with pytest.raises(RuntimeError, match="evaluate_actions"):
            env.evaluate_actions(np.zeros((2, n, 2), dtype=np.float32))
        env.evaluate_actions(act)   # a tensor on the env's device is accepted
        monkeypatch.undo()
    else:
        with pytest.raises(RuntimeError, match="evaluate_actions"):
            with torch.cuda.graph(torch.cuda.CUDAGraph()):
                env.evaluate_actions(torch.zeros((2, n, 2)))
    env.check_errors()
    env.close(); limited.close()


# ---- CPU: host emulation ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("robot", ["point", "car"])
@pytest.mark.parametrize("H,discount", [(1, 1.0), (2, 0.99), (17, 1.0), (17, 0.99)])
def test_matches_twin_hostemu(robot, H, discount):
    run_matches_twin("hostemu", robot, 0, "mixed", H, discount, n=7, warm=40)


@pytest.mark.parametrize("robot", ["point", "car"])
def test_gremlins_and_unsupervised_hostemu(robot):
    run_matches_twin("hostemu", robot, 2, "mixed", 4, 0.99, n=7, warm=30)
    run_matches_twin("hostemu", robot, 0, "unsupervised", 4, 0.99, n=4, warm=30)


@pytest.mark.parametrize("robot", ["point", "car"])
def test_physics_error_stops_the_sums_hostemu(robot):
    run_physics_error_stops_the_sums("hostemu", robot)


def test_goal_resample_inside_horizon_hostemu():
    run_goal_resample_inside_horizon("hostemu")


def test_outputs_follow_copy_outputs_hostemu():
    run_outputs_follow_copy_outputs("hostemu")


def test_refusals_hostemu(monkeypatch):
    run_refusals("hostemu", monkeypatch)


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["point", "car"])
@pytest.mark.parametrize("gremlins", [0, 2])
@pytest.mark.parametrize("tasks", ["mixed", "unsupervised"])
@pytest.mark.parametrize("H,discount", [(1, 1.0), (2, 0.99), (17, 1.0), (17, 0.99)])
def test_matches_twin_cuda(robot, gremlins, tasks, H, discount):
    run_matches_twin("cuda", robot, gremlins, tasks, H, discount, n=700, warm=300)


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["point", "car"])
def test_physics_error_stops_the_sums_cuda(robot):
    run_physics_error_stops_the_sums("cuda", robot)


@pytest.mark.gpu
def test_goal_resample_inside_horizon_cuda():
    run_goal_resample_inside_horizon("cuda")


@pytest.mark.gpu
def test_outputs_follow_copy_outputs_cuda():
    run_outputs_follow_copy_outputs("cuda")


@pytest.mark.gpu
def test_refusals_cuda(monkeypatch):
    run_refusals("cuda", monkeypatch)


@pytest.mark.gpu
def test_fullsize_point_matches_twin():
    """65,536 point go_to_goal environments late in their episodes, H = 16."""
    run_matches_twin("cuda", "point", 0, "go_to_goal", 16, 0.99, n=65536, warm=300)


@pytest.mark.gpu
@pytest.mark.parametrize("H", [1, 16])
def test_graphed_round_matches_eager(H):
    """copy_envs (K copies of every live environment) + evaluate_actions in one CUDA graph, replayed with refilled
    candidates while the live batch moves on: bit-identical to an eager planning batch issuing the same calls."""
    N, K, seed = 64, 16, 41
    env = make_env("cuda", N, [MIXED[e % len(MIXED)] for e in range(N)], seed, {"action_noise": 0.01}, max_episode_steps=50)
    plans = [make_env("cuda", N * K, "go_to_goal", seed + 1, {"action_noise": 0.0}, copy_outputs=False) for _ in range(2)]
    src_of = torch.arange(N * K, device="cuda", dtype=torch.int32) // K
    cand = torch.zeros((H, N * K, 2), device="cuda")

    def round_(plan):
        plan.copy_envs(src_of, source=env)
        return plan.evaluate_actions(cand, 0.97)

    g = torch.Generator(device="cuda").manual_seed(seed)
    round_(plans[0])   # warm-up
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = round_(plans[0])
    for r in range(5):
        cand.copy_(torch.rand((H, N * K, 2), device="cuda", generator=g) * 2 - 1)
        graph.replay()
        eager = [t.clone() for t in round_(plans[1])]
        for name, x, y in zip(("obs", "ret", "cost", "length"), out, eager):
            assert_same_bits(x, y, f"{name} round {r}")
        assert_same_state(plans[0], plans[1], f"round {r}")
        best = (out[1] - out[2]).view(N, K).argmax(1)
        env.step(cand[0].view(N, K, 2)[torch.arange(N, device="cuda"), best])
    assert float(out[1].abs().sum()) > 0.0
    env.check_errors()
    for p in plans:
        p.check_errors()
