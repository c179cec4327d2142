#!/usr/bin/env python
"""Eager against CUDA-graphed training-loop step: a fixed-weight policy MLP computes the actions from the previous
observation, then env.step with auto-reset (copy_outputs=False).  The graphed form records that policy + step once
(torch.cuda.graph) and replays it every step.  Point go_to_goal at several batch sizes; the two forms alternate in one
run, each timed with device events over windows of at least --seconds after a warm-up.  Writes a JSON file with the
card's name and power limit beside the numbers.

    python tools/probe_cuda_graphs.py --out profiles/cuda_graphs_probe.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import safe_adaptation_gym_b200 as sag  # noqa: E402


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


def time_window(run_one, seconds, warmup):
    """Seconds per step of run_one(), from device events around a window of at least `seconds`."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warmup):
        run_one()
    e0.record()
    for _ in range(warmup):
        run_one()
    e1.record()
    e1.synchronize()
    per = e0.elapsed_time(e1) * 1e-3 / warmup
    iters = max(warmup, int(seconds / per) + 1)
    e0.record()
    for _ in range(iters):
        run_one()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / iters, iters


def probe(n, seconds, reps, warmup):
    env = sag.make("point", "go_to_goal", seed=666, num_envs=n, device="cuda:0", max_episode_steps=1000, copy_outputs=False)
    torch.manual_seed(0)
    policy = torch.nn.Sequential(torch.nn.Linear(env.obs_dim, 64), torch.nn.Tanh(), torch.nn.Linear(64, 2),
                                 torch.nn.Tanh()).cuda()
    obs_buf = env.observation.clone()

    def loop_step():
        obs = env.step(policy(obs_buf))[0]
        obs_buf.copy_(obs)

    with torch.no_grad():
        side = torch.cuda.Stream()   # warm-up outside the capture (library handles, kernel loading)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                loop_step()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loop_step()
        rows = []
        for r in range(reps):
            for mode, fn in (("eager", loop_step), ("graph", graph.replay)):
                dt, iters = time_window(fn, seconds, warmup)
                rows.append({"rep": r, "mode": mode, "us_per_step": dt * 1e6, "env_steps_per_s": n / dt, "steps": iters})
        env.check_errors()
    env.close()
    med = {}
    for mode in ("eager", "graph"):
        v = sorted(x["us_per_step"] for x in rows if x["mode"] == mode)
        med[mode] = v[len(v) // 2]
    return {"n_envs": n, "median_us_per_step": med, "speedup_median": med["eager"] / med["graph"],
            "spread_us": {m: [min(x["us_per_step"] for x in rows if x["mode"] == m),
                              max(x["us_per_step"] for x in rows if x["mode"] == m)] for m in med},
            "windows": rows}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--sizes", default="1024,8192,65536")
    ap.add_argument("--seconds", type=float, default=1.0, help="length of each timed window")
    ap.add_argument("--reps", type=int, default=3, help="eager / graph alternations per size")
    ap.add_argument("--warmup", type=int, default=50, help="untimed steps before each window")
    ap.add_argument("--out", default=None, help="JSON file to write (the JSON is printed either way)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_cuda_graphs: needs a CUDA device")
    res = {"probe": "policy MLP + env.step (auto-reset, copy_outputs=False): eager vs one CUDA graph per step",
           "task": "point go_to_goal, max_episode_steps=1000",
           "gpu": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(),
           "torch": torch.__version__, "cuda": torch.version.cuda,
           "timing": "CUDA events around windows of >= %.2f s after %d warm-up steps; %d alternations" % (a.seconds, a.warmup, a.reps),
           "sizes": [probe(int(n), a.seconds, a.reps, a.warmup) for n in a.sizes.split(",")]}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
