#!/usr/bin/env python
"""Cost of per-environment task switches (env.set_next_task), on the GPU, with CUDA events:

- the sparse auto-reset (k of 65,536 point go_to_goal environments carry the NEEDS_RESET flag, as tools/probe_reset.py)
  without and with a task queued for each of them (the same task id: a fresh Task instance, same layout work);
- the whole-batch reset, without and with a task queued for every environment;
- a training loop recorded in one CUDA graph: policy MLP + env.step (auto-reset), against policy MLP + next-task ids
  computed by torch ops from the episode counters (a per-environment schedule, 3 episodes per task) + set_next_task +
  env.step; staggered 1000-step episodes, random_bound on (so the armed loop also refreshes the bound).  The two
  graphs alternate, each timed over windows of at least --seconds.

Writes a JSON file with the card's name and power limit beside the numbers.

    python tools/probe_task_switch.py --out profiles/task_switch_probe.json
"""
import argparse
import ctypes as C
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import safe_adaptation_gym_b200 as sag  # noqa: E402
from probe_cuda_graphs import power_limit_w, time_window  # noqa: E402
from safe_adaptation_gym_b200.benchmark import TASK_IDS  # noqa: E402


def _stats(ts):
    ts = sorted(ts)
    return {"median": round(ts[len(ts) // 2], 1), "min": round(ts[0], 1), "max": round(ts[-1], 1)}


def _timed(fn, stream):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    fn()
    b.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3


def probe_resets(reps):
    n = 65536
    dev = torch.device("cuda:0")
    env = sag.make("point", "go_to_goal", seed=666, num_envs=n, device=dev)
    L, h, p = env._lib, env._h, env._p
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)
    wr = torch.zeros(n, dtype=torch.uint8, device=dev)
    gtg = TASK_IDS["go_to_goal"]
    out = {"sparse_auto_reset_us": {}, "whole_batch_reset_us": {}}
    for k in (1, 64, 256):
        idx = (torch.arange(k, device=dev) * (n // k)).long()
        row = {}
        for mode in ("no_switch", "switch", "no_switch_again"):
            ts = []
            for _ in range(reps):
                fl = env.get_field("flags")
                fl[idx] |= 4
                env.set_field("flags", fl)
                if mode == "switch":
                    nxt = torch.full((n,), -1, dtype=torch.int32, device=dev)
                    nxt[idx] = gtg
                    L.check(L.L.sag_set_next_tasks(h, p(nxt), sp))
                torch.cuda.synchronize()
                ts.append(_timed(lambda: L.check(L.L.sag_reset_obs(h, None, 1, 0, p(env._obs), p(wr), sp)), stream))
                assert int(wr.sum()) == k
                if mode == "switch":
                    assert int((env.get_field("next_task")[:n] != -1).sum()) == 0
            row[mode] = _stats(ts)
        out["sparse_auto_reset_us"]["%d of %d" % (k, n)] = row
    all_q = torch.full((n,), gtg, dtype=torch.int32, device=dev)
    for mode in ("no_switch", "switch", "no_switch_again"):
        ts = []
        for _ in range(reps):
            if mode == "switch":
                L.check(L.L.sag_set_next_tasks(h, p(all_q), sp))
            torch.cuda.synchronize()
            ts.append(_timed(lambda: L.check(L.L.sag_reset(h, None, 0, 0, sp)), stream))
        out["whole_batch_reset_us"][mode] = _stats(ts)
    env.check_errors()
    env.close()
    return out


def probe_loop(n, seconds, reps, warmup):
    cycle = torch.tensor([TASK_IDS[x] for x in ("go_to_goal", "push_box", "press_buttons", "collect")], dtype=torch.int32)
    res = {}
    graphs = {}
    envs = []
    for mode in ("plain", "armed"):
        env = sag.make("point", "go_to_goal", seed=666, num_envs=n, device="cuda:0", max_episode_steps=1000,
                       copy_outputs=False, config={"random_bound": True})
        ti = env.get_field("task_i32")
        ti[6, :n] = torch.arange(n, device="cuda", dtype=torch.int32) % 1000   # staggered episodes
        env.set_field("task_i32", ti)
        torch.manual_seed(0)
        policy = torch.nn.Sequential(torch.nn.Linear(env.obs_dim, 64), torch.nn.Tanh(), torch.nn.Linear(64, 2),
                                     torch.nn.Tanh()).cuda()
        schedule = cycle[torch.randint(0, len(cycle), (n, 8))].cuda()
        obs_buf = env.observation.clone()

        def loop_step(env=env, policy=policy, obs_buf=obs_buf, schedule=schedule, armed=(mode == "armed")):
            act = policy(obs_buf)
            if armed:
                nxt = env.get_field("task_i32")[8, :env.num_envs].long() + 1   # the next episode's number
                ids = schedule.gather(1, ((nxt // 3) % schedule.shape[1])[:, None])[:, 0]
                env.set_next_task(torch.where(nxt % 3 == 0, ids, torch.full_like(ids, -1)))
            obs_buf.copy_(env.step(act)[0])

        with torch.no_grad():
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    loop_step()
            torch.cuda.current_stream().wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                loop_step()
        graphs[mode] = g
        envs.append(env)
    rows = []
    with torch.no_grad():
        for r in range(reps):
            for mode in ("plain", "armed"):
                dt, iters = time_window(graphs[mode].replay, seconds, warmup)
                rows.append({"rep": r, "mode": mode, "us_per_step": dt * 1e6, "env_steps_per_s": n / dt, "steps": iters})
    for env in envs:
        env.check_errors()
    switched = int((envs[1].get_field("task_i32")[0, :n] != TASK_IDS["go_to_goal"]).sum())
    for env in envs:
        env.close()
    med = {}
    for mode in ("plain", "armed"):
        v = sorted(x["us_per_step"] for x in rows if x["mode"] == mode)
        med[mode] = v[len(v) // 2]
    res = {"n_envs": n, "median_us_per_step": med, "armed_over_plain": med["armed"] / med["plain"],
           "spread_us": {m: [min(x["us_per_step"] for x in rows if x["mode"] == m),
                             max(x["us_per_step"] for x in rows if x["mode"] == m)] for m in med},
           "envs_not_on_their_first_task_at_the_end": switched, "windows": rows}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--sizes", default="1024,8192,65536")
    ap.add_argument("--seconds", type=float, default=1.0, help="length of each timed window of the graphed loops")
    ap.add_argument("--reps", type=int, default=3, help="plain / armed alternations per size")
    ap.add_argument("--warmup", type=int, default=50, help="untimed steps before each window")
    ap.add_argument("--reset-reps", type=int, default=9, help="timed resets per reset case")
    ap.add_argument("--out", default=None, help="JSON file to write (the JSON is printed either way)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_task_switch: needs a CUDA device")
    res = {"probe": "per-environment task switches: resets with and without queued tasks; graphed policy + step loop "
                    "with and without set_next_task",
           "gpu": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(),
           "torch": torch.__version__, "cuda": torch.version.cuda,
           "resets": {"what": "65,536 point go_to_goal environments; CUDA events around one sag_reset_obs(only_flagged=1) "
                              "(sparse) or sag_reset (whole batch); median / min / max of %d; 'switch' = every reset "
                              "environment has the same task queued (fresh Task instance)" % a.reset_reps,
                      **probe_resets(a.reset_reps)},
           "graphed_loop": {"what": "policy MLP (+ next-task ids by torch ops + set_next_task) + env.step with auto-reset, "
                                    "one CUDA graph per step, max_episode_steps=1000 staggered, random_bound; CUDA events "
                                    "around windows of >= %.2f s after %d warm-up steps; %d alternations"
                                    % (a.seconds, a.warmup, a.reps),
                            "sizes": [probe_loop(int(n), a.seconds, a.reps, a.warmup) for n in a.sizes.split(",")]}}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
