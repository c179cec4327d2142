#!/usr/bin/env python
"""What scoring candidate actions with env.evaluate_actions saves, on the GPU, with CUDA events:

(a) per-step time of a horizon of H = 16 steps from the same state, sag_evaluate_actions (15 observation-free kernel
    pairs with the accumulating epilogue, then one pair that also writes the observation) against 16 sag_step calls
    (the existing pair), for
      - 65,536 point go_to_goal environments early (step 10), in the middle (300) and late (600) in their episodes,
      - 32,768 car go_to_goal environments at step 300,
    the states reached with a uniform random policy.  Before every timed horizon the working batch takes the saved
    state again (copy_envs, outside the event pair), so every horizon starts from the same state;
(b) the README's lookahead round at N = 1,024, K = 64, H = 16, each form recorded as one CUDA graph: copy_envs + the
    hand-written loop of env.step calls accumulating return and cost in torch, against copy_envs + evaluate_actions.

Each number is the median of 3 windows of at least --seconds, the two forms alternated.  Writes a JSON file with the
card's name and power limit beside the numbers.

    python tools/probe_evaluate_actions.py --out profiles/evaluate_actions_probe.json
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

H = 16


def _p(t):
    return C.c_void_p(t.data_ptr())


def timed_windows(forms, restore, seconds, chunk=8):
    """{name: [3 windows of mean event time per call, us]}; the forms alternate window by window.  restore() runs
    before every timed call, outside its event pair."""
    out = {name: [] for name in forms}
    for _ in range(3):
        for name, fn in forms.items():
            total, calls = 0.0, 0
            while total < seconds:
                evs = []
                for _ in range(chunk):
                    restore()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    fn()
                    b.record()
                    evs.append((a, b))
                evs[-1][1].synchronize()
                total += sum(a.elapsed_time(b) for a, b in evs) * 1e-3
                calls += chunk
            out[name].append(round(total / calls * 1e6, 1))
    return out


def probe_pair(robot, n, phases, seconds):
    dev = torch.device("cuda:0")
    live = sag.make(robot, "go_to_goal", seed=5, num_envs=n, device=dev, copy_outputs=False)
    work = sag.make(robot, "go_to_goal", seed=6, num_envs=n, device=dev, copy_outputs=False, config={"action_noise": 0.0})
    snap = sag.make(robot, "go_to_goal", seed=6, num_envs=n, device=dev, copy_outputs=False, config={"action_noise": 0.0})
    L = work._lib
    g = torch.Generator(device=dev).manual_seed(1)
    idx = torch.arange(n, device=dev, dtype=torch.int32)
    act = torch.rand((H, n, 2), device=dev, generator=g) * 2 - 1
    obs = torch.empty((n, work.obs_dim), device=dev)
    rew = torch.empty((n,), dtype=torch.float64, device=dev)
    cost8, done8 = torch.empty((n,), dtype=torch.uint8, device=dev), torch.empty((n,), dtype=torch.uint8, device=dev)
    ret, cost = torch.empty((n,), dtype=torch.float64, device=dev), torch.empty((n,), dtype=torch.float64, device=dev)
    length = torch.empty((n,), dtype=torch.int32, device=dev)
    stream = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731

    def steps():
        for h in range(H):
            L.check(L.L.sag_step(work._h, _p(act[h]), _p(obs), _p(rew), None, _p(cost8), _p(done8), stream()))

    def evaluate():
        L.check(L.L.sag_evaluate_actions(work._h, H, _p(act), C.c_double(1.0), _p(obs), _p(ret), 1, _p(cost), _p(length),
                                         stream()))

    res, done_steps = [], 0
    for phase in phases:
        while done_steps < phase:
            live.step(torch.rand((n, 2), device=dev, generator=g) * 2 - 1)
            done_steps += 1
        snap.copy_envs(idx, source=live)
        restore = lambda: work.copy_envs(idx, source=snap)  # noqa: E731
        # same outputs from both forms at this state (a check of the measured paths, not a test)
        restore(); steps(); o1, r1 = obs.clone(), rew.clone()
        restore(); evaluate()
        same_obs = bool(torch.equal(o1.view(torch.int32), obs.view(torch.int32)))
        for _ in range(3):
            restore(); steps(); restore(); evaluate()
        torch.cuda.synchronize()
        busy = int((snap.get_field("task_i32")[9, :n] != 0).sum())
        w = timed_windows({"step_pair": steps, "evaluate": evaluate}, restore, seconds)
        med = {k: sorted(v)[1] for k, v in w.items()}
        res.append({"robot": robot, "n": n, "episode_step": phase, "H": H, "envs_with_moving_bodies": busy,
                    "horizon_us_windows": w, "horizon_us_median": med,
                    "per_step_us": {k: round(v / H, 2) for k, v in med.items()},
                    "evaluate_over_step": round(med["evaluate"] / med["step_pair"], 3),
                    "last_obs_identical": same_obs})
        work.check_errors()
    for env in (live, work, snap):
        env.close()
    return res


def probe_round(seconds):
    N, K = 1024, 64
    dev = torch.device("cuda:0")
    env = sag.make("point", "go_to_goal", seed=3, num_envs=N, device=dev, max_episode_steps=1000)
    plans = [sag.make("point", "go_to_goal", seed=4, num_envs=N * K, device=dev, copy_outputs=False,
                      config={"action_noise": 0.0}) for _ in range(2)]
    src_of = torch.arange(N * K, device=dev, dtype=torch.int32) // K
    g = torch.Generator(device=dev).manual_seed(0)
    cand = torch.rand((H, N * K, 2), device=dev, generator=g) * 2 - 1
    acc = torch.zeros((2, N * K), dtype=torch.float64, device=dev)
    out = {}

    def hand():
        plans[0].copy_envs(src_of, source=env)
        acc.zero_()
        for h in range(H):
            _, r, _, info = plans[0].step(cand[h])
            acc[0] += r
            acc[1] += info["cost"]

    def scored():
        plans[1].copy_envs(src_of, source=env)
        out["r"] = plans[1].evaluate_actions(cand)

    graphs = {}
    for name, fn in (("hand_loop", hand), ("evaluate_actions", scored)):
        fn()
        torch.cuda.synchronize()
        graphs[name] = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graphs[name]):
            fn()
    for gr in graphs.values():
        gr.replay()
    torch.cuda.synchronize()
    _, ret, cost, length = out["r"]
    full = length == H   # the hand loop does not stop at a physics error
    same = bool(torch.equal(acc[0][full], ret[full]) and torch.equal(acc[1][full], cost[full]))
    windows = {k: [] for k in graphs}
    for _ in range(3):
        for name, gr in graphs.items():
            s, _ = time_window(gr.replay, seconds, 3)
            windows[name].append(round(s * 1e6, 1))
    med = {k: sorted(v)[1] for k, v in windows.items()}
    for p in plans:
        p.check_errors()
    return {"N": N, "K": K, "H": H, "env_steps_per_round": N * K * H, "round_us_windows": windows,
            "round_us_median": med, "speedup": round(med["hand_loop"] / med["evaluate_actions"], 3),
            "sums_match_hand_loop": same, "environments_ended_early": int((~full).sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/evaluate_actions_probe.json")
    ap.add_argument("--seconds", type=float, default=1.0)
    a = ap.parse_args()
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(),
           "l2": "the working batch is rewritten from the saved state (copy_envs) before every timed horizon",
           "pair": probe_pair("point", 65536, (10, 300, 600), a.seconds) + probe_pair("car", 32768, (300,), a.seconds)}
    res["lookahead_round"] = probe_round(a.seconds)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
