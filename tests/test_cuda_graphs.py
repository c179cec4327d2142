"""env.step / env.rollout / env.observation recorded in a CUDA graph (torch.cuda.graph) and replayed, against an eager
twin created with the same seed, tasks and config and stepped with the same actions: outputs and state bit-identical.
The CPU tests check that the synchronising methods refuse to run while a capture is open (host-emulated library)."""
import numpy as np
import pytest
import torch

from common import make_env
from safe_adaptation_gym_b200 import tasks
from safe_adaptation_gym_b200.benchmark import TASKS

T = 7  # max_episode_steps of the short-episode cases
MIXED = ["go_to_goal", "press_buttons", "push_box", "collect", "catch_goal", "haul_box", "go_to_goal_scarce", "roll_rod"]


def _twins(n, task_names, seed, robot="point", config=None, **kw):
    return (make_env("cuda", n, task_names, seed, config, robot=robot, **kw),
            make_env("cuda", n, task_names, seed, config, robot=robot, **kw))


def _set_bodies_moving(envs):
    """Give every object slot a small velocity (the same in both twins) and rebuild the derived moving-body mask, so that
    every environment with a movable body is on the contact kernel's work list from the first step on."""
    for env in envs:
        objs = env.get_field("objects")
        objs[3] = 0.2
        env.set_field("objects", objs)
        _ = env.observation


def _snap(out):
    obs, rew, done, info = out
    s = [obs, rew, done, info["cost"], info["bound"]]
    if "truncated" in info:
        s.append(info["truncated"])
    return [t.clone() for t in s]


def _assert_same(a, b, msg):
    assert len(a) == len(b), msg
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x.cpu().numpy(), y.cpu().numpy(), err_msg=msg)


def _assert_same_state(ga, eb):
    for name in ga._FIELDS:
        np.testing.assert_array_equal(ga.get_field(name).cpu().numpy(), eb.get_field(name).cpu().numpy(), err_msg=name)


def _moving(env):
    return int((env.get_field("task_i32")[9, :env.num_envs] != 0).sum())


def _run_step_graph(ge, ee, k, replays, rng):
    """Capture k steps of `ge` (actions from a static device tensor), replay them, step `ee` eagerly with the same
    actions; compare every step.  Returns the largest number of environments with a moving body seen
    after a replay (they are on the next step's work list)."""
    n = ge.num_envs
    act = torch.zeros((k, n, 2), dtype=torch.float32, device="cuda")
    _assert_same(_snap(ge.step(act[0])), _snap(ee.step(act[0])), "warm-up step")   # loads every kernel of the step
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        snaps = [_snap(ge.step(act[i])) for i in range(k)]
    most = 0
    for r in range(replays):
        act.copy_(torch.from_numpy(rng.uniform(-1, 1, (k, n, 2)).astype(np.float32)))
        graph.replay()
        for i in range(k):
            _assert_same(snaps[i], _snap(ee.step(act[i])), f"replay {r} step {i} of the graph")
        most = max(most, _moving(ge))
    torch.cuda.synchronize()
    return most


CASES = [
    pytest.param("push_box", "point", 0, True, id="push_box-point-copy"),
    pytest.param("haul_box", "car", 0, False, id="haul_box-car-views"),
    pytest.param("mixed", "point", 2, False, id="mixed-pointG-views"),
    pytest.param("mixed", "car", 2, True, id="mixed-carG-copy"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 3])
@pytest.mark.parametrize("task,robot,gremlins,copy_outputs", CASES)
def test_step_graph_matches_eager(task, robot, gremlins, copy_outputs, k):
    """Graphs of 1, 2 and 3 steps replayed over more than three short episodes (auto-reset inside the graph).  A graph of
    an odd number of steps is the case a host-side choice of the work-list counter set gets wrong."""
    n = 256
    names = [MIXED[e % len(MIXED)] for e in range(n)] if task == "mixed" else task
    cfg = {"num_gremlins": gremlins} if gremlins else None
    ge, ee = _twins(n, names, 31 + k, robot, cfg, max_episode_steps=T, copy_outputs=copy_outputs)
    _set_bodies_moving((ge, ee))
    replays = -(-(3 * T + 2) // k)
    most = _run_step_graph(ge, ee, k, replays, np.random.RandomState(k))
    assert most > 0   # the contact kernel's work list was not empty during the replays
    _assert_same_state(ge, ee)


@pytest.mark.gpu
@pytest.mark.parametrize("copy_outputs", [True, False])
def test_step_graph_without_episode_limit(copy_outputs):
    ge, ee = _twins(128, "push_box", 41, copy_outputs=copy_outputs)
    _set_bodies_moving((ge, ee))
    assert _run_step_graph(ge, ee, 3, 10, np.random.RandomState(0)) > 0
    _assert_same_state(ge, ee)


class _Policy:
    """Fixed-weight two-layer MLP, observation -> action in [-1, 1].  Written with broadcast products and sums (no
    matrix-multiply library call) so that its arithmetic is the same inside and outside a graph."""

    def __init__(self, obs_dim, hidden=16, seed=0):
        g = torch.Generator().manual_seed(seed)
        self.w1 = (torch.randn((obs_dim, hidden), generator=g) / obs_dim ** 0.5).cuda()
        self.w2 = (torch.randn((hidden, 2), generator=g) / hidden ** 0.5).cuda()

    def __call__(self, obs):
        h = torch.tanh((obs[:, :, None] * self.w1[None]).sum(1))
        return torch.tanh((h[:, :, None] * self.w2[None]).sum(1))


@pytest.mark.gpu
@pytest.mark.parametrize("copy_outputs", [True, False])
def test_policy_and_step_in_one_graph(copy_outputs):
    n = 256
    ge, ee = _twins(n, MIXED * (n // len(MIXED)), 43, max_episode_steps=T, copy_outputs=copy_outputs)
    _set_bodies_moving((ge, ee))
    pi = _Policy(ge.obs_dim)
    g_obs, e_obs = ge.observation.clone(), ee.observation.clone()
    _assert_same(_snap(ge.step(pi(g_obs))), _snap(ee.step(pi(e_obs))), "warm-up step")
    g_obs.copy_(ge.observation)
    e_obs.copy_(ee.observation)
    _assert_same([g_obs], [e_obs], "observation")
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = ge.step(pi(g_obs))
        g_obs.copy_(out[0])
        snap = _snap(out)
    for t in range(3 * T + 2):
        graph.replay()
        want = ee.step(pi(e_obs))
        e_obs.copy_(want[0])
        _assert_same(snap, _snap(want), f"step {t}")
    _assert_same_state(ge, ee)


@pytest.mark.gpu
def test_rollout_and_observation_graph():
    ge, ee = _twins(256, "push_box", 47, robot="car")
    _set_bodies_moving((ge, ee))
    _assert_same(list(ge.rollout(1)[:3]), list(ee.rollout(1)[:3]), "warm-up rollout")
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        obs, rew, done, info = ge.rollout(4)
        snap = [obs.clone(), rew.clone(), done.clone(), info["cost"].clone(), ge.observation]
    for r in range(6):
        graph.replay()
        obs, rew, done, info = ee.rollout(4)
        _assert_same(snap, [obs, rew, done, info["cost"], ee.observation], f"replay {r}")
    _assert_same_state(ge, ee)


@pytest.mark.gpu
def test_graph_follows_seed_and_state_dict():
    n = 256
    ge, ee = _twins(n, "push_box", 53, max_episode_steps=T)
    _set_bodies_moving((ge, ee))
    act = torch.zeros((n, 2), device="cuda")
    _assert_same(_snap(ge.step(act)), _snap(ee.step(act)), "warm-up step")
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        snap = _snap(ge.step(act))
    rng = np.random.RandomState(5)

    def run(steps, tag):
        for t in range(steps):
            act.copy_(torch.from_numpy(rng.uniform(-1, 1, (n, 2)).astype(np.float32)))
            graph.replay()
            _assert_same(snap, _snap(ee.step(act)), f"{tag} step {t}")

    run(5, "before")
    sd = ee.state_dict()
    run(T + 3, "saved")
    for env in (ge, ee):
        env.seed(1234)        # new Philox key: action noise and auto-reset layouts
    run(T + 3, "reseeded")
    for env in (ge, ee):
        env.load_state_dict(sd)   # back to the saved state and the saved key
    run(T + 3, "restored")
    _assert_same_state(ge, ee)


@pytest.mark.gpu
@pytest.mark.parametrize("copy_outputs", [True, False])
def test_graph_follows_set_task_random_bound(copy_outputs):
    n = 128
    ge, ee = _twins(n, "go_to_goal", 59, config={"random_bound": True}, max_episode_steps=T, copy_outputs=copy_outputs)
    act = torch.zeros((n, 2), device="cuda")
    _assert_same(_snap(ge.step(act)), _snap(ee.step(act)), "warm-up step")
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = ge.step(act)
        snap = _snap(out)
    graph.replay()
    _assert_same(snap, _snap(ee.step(act)), "before set_task")
    before = snap[4].clone()
    for env in (ge, ee):
        env.set_task([TASKS["push_box"]()] * n)   # a new Task instance: new bounds
    for t in range(T + 2):
        graph.replay()
        want = ee.step(act)
        _assert_same(snap, _snap(want), f"after set_task step {t}")
        np.testing.assert_array_equal(out[3]["bound"].cpu().numpy(), want[3]["bound"].cpu().numpy())
    assert not torch.equal(snap[4], before)   # the exported bound followed the new draw
    _assert_same_state(ge, ee)


@pytest.mark.gpu
def test_full_size_episode_from_one_step_graph():
    """65,536 point go_to_goal environments, one whole 1000-step episode and 20 steps of the next."""
    n, steps = 65536, 1020
    ge, ee = _twins(n, "go_to_goal", 61, max_episode_steps=1000, copy_outputs=False)
    act = torch.zeros((n, 2), device="cuda")
    _assert_same(_snap(ge.step(act)), _snap(ee.step(act)), "warm-up step")
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        snap = _snap(ge.step(act))
    g = torch.Generator(device="cuda").manual_seed(7)
    check = set(range(0, steps, 97)) | {997, 998, 999, 1000, 1001, steps - 1}
    for t in range(1, steps):
        act.uniform_(-1, 1, generator=g)
        graph.replay()
        want = ee.step(act)
        if t in check:
            _assert_same(snap, _snap(want), f"step {t}")
    _assert_same_state(ge, ee)
    assert int(ge.get_field("task_i32")[8, :n].min()) >= 1   # every environment is past its first episode


# ---- CPU: the methods that synchronise refuse to be recorded -----------------------------------------------------------
def _hostemu_env(**kw):
    return make_env("hostemu", 4, "go_to_goal", 3, **kw)


def test_synchronising_methods_raise_under_capture(monkeypatch):
    env = _hostemu_env()
    sd = env.state_dict()
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: True)
    calls = {
        "reset": lambda: env.reset(),
        "reset_envs": lambda: env.reset_envs(np.ones(4, dtype=bool)),
        "set_task": lambda: env.set_task(tasks.PushBox()),
        "seed": lambda: env.seed(5),
        "set_field": lambda: env.set_field("flags", env.get_field("flags")),
        "load_state_dict": lambda: env.load_state_dict(sd),
        "check_errors": lambda: env.check_errors(),
        "state_dict": lambda: env.state_dict(),
    }
    for name, call in calls.items():
        with pytest.raises(RuntimeError, match=name):
            call()
    with pytest.raises(RuntimeError, match="action"):
        env.step(np.zeros((4, 2), dtype=np.float32))
    obs, rew, done, info = env.step(torch.zeros((4, 2)))   # a tensor already on the env's device is accepted
    assert tuple(obs.shape) == (4, env.obs_dim)


def test_bound_is_updated_in_place():
    """A graph bakes the address of the exported bound in: set_task / load_state_dict must write into the same tensor."""
    env = _hostemu_env(config={"random_bound": True})
    bound = env._bound
    first = bound.clone()
    sd = env.state_dict()
    env.set_task(tasks.GoToGoal())
    assert env._bound is bound and not torch.equal(bound, first)
    env.load_state_dict(sd)
    assert env._bound is bound and torch.equal(bound, first)
