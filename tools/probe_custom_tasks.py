#!/usr/bin/env python
"""What running a user-defined task costs, on the GPU, with CUDA events.

65,536 point environments, uniform random actions, action noise 0:
  (a) a user-defined task whose obstacles and placement extents equal GoToGoal's (so it runs the *C kernel set with the
      same trajectories as GoToGoal, same seed), against GoToGoal itself: the mean step time over 20 steps starting at
      episode steps 10, 300 and 600;
  (b) the same for a GoToGoal with 15 hazards and 6 vases (its own trajectories);
  (c) the whole-batch reset time of each of the four batches (median of 5).
The batches are stepped side by side (alternating every step), each step is timed with device events.  (a) and (b) are
repeated over --repeats episodes (new layouts, the same for GoToGoal and its custom twin): the JSON has every repeat,
and for (a) the ratio custom / GoToGoal per repeat, so that a difference can be read against the spread.
Writes a JSON file with the card's name and power limit beside the numbers.

    python tools/probe_custom_tasks.py --out profiles/custom_tasks_probe.json
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import safe_adaptation_gym_b200 as sag  # noqa: E402
from safe_adaptation_gym_b200 import tasks  # noqa: E402
from probe_cuda_graphs import power_limit_w  # noqa: E402


class SameAsGoToGoal(tasks.GoToGoal):
    @property
    def obstacles(self):
        return [9, 10, 0, 1]

    @property
    def placement_extents(self):
        return (-2.0, -2.0, 2.0, 2.0)


class HardGoToGoal(tasks.GoToGoal):
    @property
    def obstacles(self):
        return [15, 6, 0, 1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--out", default="profiles/custom_tasks_probe.json")
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args()
    n = a.n
    batches = {}
    for name, task, custom_id in (("go_to_goal", tasks.GoToGoal(), False), ("custom_same_as_go_to_goal", SameAsGoToGoal(), True),
                                  ("go_to_goal_for_hard", tasks.GoToGoal(), False), ("custom_15_hazards_6_vases", HardGoToGoal(), True)):
        env = sag.make("point", "go_to_goal", seed=a.seed, config={"action_noise": 0.0}, num_envs=n, device="cuda:0")
        if custom_id:
            # the spec equal to GoToGoal's would keep the registry id: define it through the C ABI to get a custom id
            from safe_adaptation_gym_b200 import _abi
            import ctypes as C
            base, ob, ext = tasks.definition(task)
            d = _abi.SagTaskDef(base.task_id, (C.c_int32 * 4)(*ob), (C.c_double * 4)(*ext))
            tid = C.c_int32()
            env._lib.check(env._lib.L.sag_define_task(env._h, C.byref(d), C.byref(tid)))
            ids = torch.full((n,), tid.value, dtype=torch.int32, device="cuda:0")
            env._lib.check(env._lib.L.sag_set_tasks(env._h, env._p(ids), env._stream()))
            env._reset_all(new_task=True)
        else:
            env.set_task(task)
        batches[name] = env
    torch.cuda.synchronize()
    # (c) whole-batch reset times (median of 5)
    reset_us = {}
    for name, env in batches.items():
        ts = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            env._lib.check(env._lib.L.sag_reset(env._h, None, 0, 0, env._stream()))
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        reset_us[name] = round(float(np.median(ts)), 1)
        env._lib.L.sag_error_flags(env._h, 1)
    # (a), (b): step times at episode steps 10, 300, 600 (all batches start a new episode together), per repeat
    g = torch.Generator(device="cuda:0").manual_seed(0)
    step_us = {name: {str(at): [] for at in (10, 300, 600)} for name in batches}
    same = True
    for _ in range(a.repeats):
        for env in batches.values():
            env.reset()
        t = 0
        for at in (10, 300, 600):
            while t < at:
                act = torch.rand((n, 2), generator=g, device="cuda:0") * 2 - 1
                for env in batches.values():
                    env.step(act)
                t += 1
            sums = {name: 0.0 for name in batches}
            for _ in range(20):
                act = torch.rand((n, 2), generator=g, device="cuda:0") * 2 - 1
                for name, env in batches.items():
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    env._lib.check(env._lib.L.sag_step(env._h, env._p(act), env._p(env._obs), env._p(env._reward), None,
                                                       env._p(env._cost), env._p(env._done), env._stream()))
                    e1.record()
                    e1.synchronize()
                    sums[name] += e0.elapsed_time(e1) * 1e3
                t += 1
            for name in batches:
                step_us[name][str(at)].append(round(sums[name] / 20, 1))
        same = same and bool(torch.equal(batches["go_to_goal"].get_field("robot"),
                                         batches["custom_same_as_go_to_goal"].get_field("robot")))
    ratio = {at: [round(c / b, 4) for c, b in zip(step_us["custom_same_as_go_to_goal"][at], step_us["go_to_goal"][at])]
             for at in step_us["go_to_goal"]}
    out = {
        "gpu": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(), "n_envs": n, "robot": "point",
        "repeats": a.repeats, "step_us_at_episode_step": step_us,
        "custom_same_over_go_to_goal_per_repeat": ratio, "whole_batch_reset_us": reset_us,
        "custom_same_spec_trajectories_identical_to_go_to_goal": same,
        "not_measured": ["car custom builds", "gremlin custom builds"],
    }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
