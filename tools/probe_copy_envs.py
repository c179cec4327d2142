#!/usr/bin/env python
"""Cost of environment copies (env.copy_envs, k_copy_envs), on the GPU, with CUDA events:

(a) sag_copy_envs alone (its two launches: k_copy_envs_fold, which settles the destinations' statistics, and the
    gather k_copy_envs), over many calls, with a 256 MiB memset between timed calls so that every call reads and writes
    HBM (outside the event pair), for
      - 65,536 -> 65,536 point environments, a random permutation of another handle (every byte read and written once);
      - 1,024 -> 65,536 broadcast, each source to 64 consecutive destinations (reads come from L2 after the first);
      - 256 -> 256, a permutation (launch-bound);
    with GB/s = bytes the copy must move / kernel time, and the share of the 6538 GB/s HBM copy peak the project
    measured on the B200 (DESIGN.md 8d);
(b) the README's lookahead round -- copy the live state of N = 1,024 environments into K = 64 copies each, then H = 16
    steps of candidate actions accumulating return and cost -- eager against one CUDA graph per round, the two
    alternated, each timed over windows of at least --seconds.

Writes a JSON file with the card's name and power limit beside the numbers.

    python tools/probe_copy_envs.py --out profiles/copy_envs_probe.json
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
from safe_adaptation_gym_b200 import _abi  # noqa: E402

HBM_COPY_PEAK_GBS = 6538.3   # measured device-to-device copy rate of the B200 (DESIGN.md 8d)


def bytes_per_env(env):
    """One environment's state: every row of every field (what a copy moves per destination)."""
    return sum(env._lib.L.sag_field_bytes(env._h, f) for f in range(_abi.F_NEXT_TASK + 1)) // env.stride


def _stats(ts):
    ts = sorted(ts)
    return {"median": round(ts[len(ts) // 2], 2), "min": round(ts[0], 2), "max": round(ts[-1], 2)}


def probe_kernel(name, n_src, n_dst, idx, reps, flush):
    dev = torch.device("cuda:0")
    src = sag.make("point", "go_to_goal", seed=1, num_envs=n_src, device=dev)
    dst = sag.make("point", "go_to_goal", seed=2, num_envs=n_dst, device=dev, config={"action_noise": 0.0})
    L = dst._lib
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)
    idx = idx.to(device=dev, dtype=torch.int32).contiguous()
    call = lambda: L.check(L.L.sag_copy_envs(dst._h, src._h, C.c_void_p(idx.data_ptr()), sp))  # noqa: E731
    for _ in range(5):
        call()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        call()
        b.record(stream)
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    ok = torch.equal(dst.get_field("objects")[:, :, :n_dst], src.get_field("objects")[:, :, idx.long()])
    dst.check_errors()
    uniq = int(torch.unique(idx[idx >= 0]).numel())
    per = bytes_per_env(dst)
    moved = n_dst * per + uniq * per   # written once, each distinct source read once
    t = _stats(ts)
    out = {"case": name, "n_src": n_src, "n_dst": n_dst, "kernel_us": t, "bytes_moved": moved,
           "bytes_per_env": per, "bytes_written": n_dst * per, "gb_per_s_median": round(moved / (t["median"] * 1e-6) / 1e9, 1),
           "share_of_hbm_copy_peak": round(moved / (t["median"] * 1e-6) / 1e9 / HBM_COPY_PEAK_GBS, 3),
           "objects_field_matches_sources": bool(ok), "launches": reps}
    src.close(); dst.close()
    return out


def probe_lookahead(seconds):
    N, K, H = 1024, 64, 16
    dev = torch.device("cuda:0")
    env = sag.make("point", "go_to_goal", seed=3, num_envs=N, device=dev, max_episode_steps=1000)
    plan = sag.make("point", "go_to_goal", seed=4, num_envs=N * K, device=dev, copy_outputs=False,
                    config={"action_noise": 0.0})
    src_of = torch.arange(N * K, device=dev, dtype=torch.int32) // K
    g = torch.Generator(device=dev).manual_seed(0)
    cand = torch.rand((H, N * K, 2), device=dev, generator=g) * 2 - 1
    ret = torch.zeros((2, N * K), dtype=torch.float64, device=dev)

    def round_():
        plan.copy_envs(src_of, source=env)
        ret.zero_()
        for h in range(H):
            _, rew, _, info = plan.step(cand[h])
            ret[0] += rew
            ret[1] += info["cost"]

    round_()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        round_()
    windows = {"eager": [], "graph": []}
    for _ in range(3):
        for mode, fn in (("eager", round_), ("graph", graph.replay)):
            s, iters = time_window(fn, seconds, 3)
            windows[mode].append(round(s * 1e6, 1))
    med = {m: sorted(v)[1] for m, v in windows.items()}
    plan.check_errors()
    return {"N": N, "K": K, "H": H, "env_steps_per_round": N * K * H, "round_us_windows": windows,
            "round_us_median": med, "graph_speedup": round(med["eager"] / med["graph"], 3),
            "planning_env_steps_per_s_graph": round(N * K * H / (med["graph"] * 1e-6), 0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/copy_envs_probe.json")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--seconds", type=float, default=1.0)
    a = ap.parse_args()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    g = torch.Generator().manual_seed(0)
    big = 65536
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(),
           "hbm_copy_peak_gb_per_s": HBM_COPY_PEAK_GBS,
           "l2": "256 MiB memset between timed launches, outside the event pair",
           "kernel": [probe_kernel("65536 -> 65536 permutation, other handle", big, big, torch.randperm(big, generator=g), a.reps, flush),
                      probe_kernel("1024 -> 65536 broadcast x64", 1024, big, torch.arange(big) // 64, a.reps, flush),
                      probe_kernel("256 -> 256 permutation, other handle", 256, 256, torch.randperm(256, generator=g), a.reps, flush)]}
    res["lookahead"] = probe_lookahead(a.seconds)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
