#!/usr/bin/env python
"""env.rollout(K) throughput (K steps enqueued in one call, Philox actions on the device)."""
import os, sys, time, torch
sys.path.insert(0, os.getcwd())
import safe_adaptation_gym_b200 as sag
env = sag.make("point", "go_to_goal", seed=666, num_envs=65536, device="cuda:0")
env.rollout(300); torch.cuda.synchronize()
t0 = time.perf_counter(); env.rollout(200); torch.cuda.synchronize(); t1 = time.perf_counter()
print("rollout(200) at steps 300-500: %.1f ms -> %.3e env-steps/s" % (1e3 * (t1 - t0), 65536 * 200 / (t1 - t0)))
