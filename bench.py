#!/usr/bin/env python
"""bench.py -- env-steps/sec of the per-step environment loop (BASELINE.json metric), whole-episode average.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port on all host cores
    python bench.py --config car_gtg_pb | haul_push_point | haul_push_car   # the other BASELINE configs
    python bench.py --steps K --dump-outputs DIR   # also write the last timed step's outputs to DIR/<name>.npy

Workload (default, N=1): BASELINE.json configs[1] -- point go_to_goal, 65,536 environments per GPU, pseudo-lidar
observation + hazard/vase/pillar cost, i.i.d. U(-1,1) actions, action_noise 0.01 (reference default), 1000-step
episodes (tests/test_safety_gym.py:78).  A "step" = one env.step over the whole batch.

The cost of a step depends on the episode phase (no robot is near anything right after a reset; ~10 % of them
are late in the episode), so the K timed steps are STRATIFIED over whole episodes: ceil(K / 1000) episodes share
them as evenly as possible, and an episode that times Ke of them does so in S = min(Ke, 20) windows of Ke/S
consecutive steps centred at (i + 1/2) * 1000 / S; the steps between the windows run untimed with the same kernels
(fast-forward), and the episode's reset (layout rejection sampling, timed with events) is added
amortised as t_reset / 1000 per step.  `value` is therefore the whole-episode average the reference arm
measures by running whole episodes.

value        : env-steps/s with actions resident in HBM, each timed step bracketed by CUDA events on the launching
               stream, L2 flushed (256 MiB memset) before every timed step.
e2e          : same metric and strata through sag_step_host (C ABI, pinned HOST buffers): H2D of the actions and
               D2H of obs/reward/cost/done inside the timed region, every step.
roofline     : algorithmic bytes per env-step (SURVEY 8d) x envs / average step duration vs the measured HBM
               copy bandwidth.
cpu_baseline : the oracle port (oracle/sag_oracle.c, pthreads) on the box's host cores, whole episodes.

--dump-outputs DIR writes what the last timed step returned (rank 0's environments): obs.npy (float32 [n, obs_dim]),
reward.npy (float64 [n]), cost.npy and done.npy (float32 [n]).  Seeds are fixed, so two builds run with the same
arguments can be compared output for output.  Above DUMP_BYTES a fixed, seeded sample of rows is written instead,
with their environment indices in env_index.npy.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

EPISODE = 1000  # tests/test_safety_gym.py:78
UNIT = "env-steps/s"
DUMP_BYTES = 60_000_000  # data budget of --dump-outputs (all files together stay under 64 MB)
# SURVEY.md 8(d): algorithmic bytes per env-step of the fused step
CONFIGS = {
    "point_gtg": dict(robot="point", tasks=["go_to_goal"], envs=65536, b_alg=2582, metric="env_steps_per_sec_point_go_to_goal",
                      workload="point go_to_goal, 65536 envs/GPU, lidar obs + hazard/vase/pillar cost, U(-1,1) actions"),
    "car_gtg_pb": dict(robot="car", tasks=["go_to_goal", "press_buttons"], envs=32768, b_alg=2918,
                       metric="env_steps_per_sec_car_go_to_goal_press_buttons",
                       workload="car go_to_goal + press_buttons (alternating envs), 32768 envs/GPU, U(-1,1) actions"),
    "haul_push_point": dict(robot="point", tasks=["haul_box", "push_box"], envs=16384, b_alg=1278,
                            metric="env_steps_per_sec_point_haul_box_push_box",
                            workload="point haul_box + push_box (alternating envs), 16384 envs/GPU, U(-1,1) actions"),
    "haul_push_car": dict(robot="car", tasks=["haul_box", "push_box"], envs=16384, b_alg=1614,
                          metric="env_steps_per_sec_car_haul_box_push_box",
                          workload="car haul_box + push_box (alternating envs), 16384 envs/GPU, U(-1,1) actions"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def strata(K):
    """[(first step, length)] of the timed windows inside one EPISODE-step episode; lengths sum to min(K, EPISODE)."""
    K = min(K, EPISODE)
    S = min(K, 20)
    out, used = [], 0
    for i in range(S):
        ln = (K * (i + 1)) // S - used
        used += ln
        centre = (i + 0.5) * EPISODE / S
        a = int(round(centre - ln / 2.0))
        a = max(a, out[-1][0] + out[-1][1] if out else 0)
        a = min(a, EPISODE - (K - used) - ln)
        out.append((a, ln))
    return out


def dump_outputs(path, obs, rew, cost, done):
    """DIR/<name>.npy of one step's outputs (device tensors, row = environment), float32 / float64, within DUMP_BYTES"""
    import numpy as np
    import torch
    arrays = {"obs": obs.float(), "reward": rew.double(), "cost": cost.float(), "done": done.float()}
    n = obs.shape[0]
    row_bytes = sum(a.element_size() * a[0].numel() for a in arrays.values())
    os.makedirs(path, exist_ok=True)
    if n * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.RandomState(0).choice(n, DUMP_BYTES // (row_bytes + 8), replace=False))
        idx = torch.from_numpy(rows).to(obs.device)
        arrays = {k: a[idx] for k, a in arrays.items()}
        np.save(os.path.join(path, "env_index.npy"), rows.astype(np.float64))
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a.cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the run (started before the warm-up)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.t_marks = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t0=None, t1=None):
        """summary over the samples taken in [t0, t1] (perf_counter; the GPU-timed region), all samples if none fall inside"""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for t, r in self.rows if t0 is None or (t0 <= t <= t1)]
        scope = "timed region"
        if not rows:
            rows, scope = [r for _, r in self.rows], "whole run (no sample fell inside the timed region)"
        sm = sorted(float(r[1]) for r in rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for k, nm in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "scope": scope}


def cpu_oracle_rate(cfg, n_envs, steps, threads, seed=666):
    """env-steps/s of the oracle port on `threads` host threads: n_envs whole-or-partial episodes from a reset."""
    import oracle as O
    tasks = cfg["tasks"]
    envs = [O.OracleEnv(cfg["robot"], tasks[i % len(tasks)], seed=seed, env_gid=i) for i in range(n_envs)]
    for e in envs:
        e.reset(0)
    t0 = time.perf_counter()
    count, sr, sc = O.batch_rollout(envs, steps, threads)
    dt = time.perf_counter() - t0
    return count / dt, count, dt


def run_reference(args, cfg, rank, world):
    """CPU arm: whole 1000-step episodes (= the same strata as the GPU arm's whole-episode average) of the oracle port."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_core = 16 if cfg["robot"] == "point" else 2
    n_envs = per_core * cores
    for _ in range(min(args.warmup, 2)):
        cpu_oracle_rate(cfg, n_envs, 20, cores)
    t_total, c_total, done = 0.0, 0, 0
    for _ in range(args.steps):
        r, c, dt = cpu_oracle_rate(cfg, n_envs, EPISODE, cores)
        t_total += dt; c_total += c; done += 1
        if t_total > 150:
            break
    value = c_total / t_total
    sample = (f"{n_envs} envs x {EPISODE} steps (whole episodes from a reset) per bench step, {done} bench steps, "
              f"oracle port (C, pthreads, {cores} threads)")
    line = {"impl": "reference", "metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_total / max(1, done), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["workload"], "episode_phase": "whole 1000-step episodes", "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "the reference's own stack (dm_control/MuJoCo) is not installable here; this arm times the CPU oracle port"}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="point_gtg", choices=sorted(CONFIGS))
    ap.add_argument("--envs-per-gpu", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--stagger", action="store_true", help="extra: episodes staggered over all 1000 phases (auto-reset every step)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write obs / reward / cost / done of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the CUDA path's outputs (--impl b200)")
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from safe_adaptation_gym_b200.benchmark import TASKS
    from safe_adaptation_gym_b200.env import BatchedSafeAdaptationGym

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    # every rank on its GPU's NUMA node with cores of its own, BEFORE any pinned allocation (pages are first-touched there)
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from probe_d2h import bind_rank_to_gpu_node
    binding = bind_rank_to_gpu_node(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    dev = torch.device("cuda", local_rank)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # before the warm-up, so that a short timed region still carries samples
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    n = args.envs_per_gpu or cfg["envs"]
    K, W = args.steps, max(3, args.warmup)
    n_ep = (K + EPISODE - 1) // EPISODE
    # episode i times K*(i+1)//n_ep - K*i//n_ep steps: exactly K timed steps in all
    ep_windows = [strata(K * (i + 1) // n_ep - K * i // n_ep) for i in range(n_ep)]
    windows = ep_windows[0]
    task_objs = [TASKS[t]() for t in cfg["tasks"]]

    def make_env():
        env = BatchedSafeAdaptationGym("xmls/%s.xml" % cfg["robot"], num_envs=n, device=dev, env_id_base=rank * n, max_episode_steps=EPISODE)  # step 1000 flags the episode as finished: its return / cost enter the per-task statistics at the reset
        env.seed(666)
        env.set_task([task_objs[(rank * n + e) % len(task_objs)] for e in range(n)])
        return env

    env = make_env()
    L, h = env._lib, env._h
    stream = torch.cuda.current_stream(dev)
    sp = C.c_void_p(stream.cuda_stream)
    p = BatchedSafeAdaptationGym._p
    launch_count = getattr(L.L, "sag_launch_count", None)

    def launches_now(hh):
        return int(launch_count(hh)) if launch_count is not None else 0

    # synthetic actions, resident in HBM: i.i.d. U(-1,1) per env per step (env.action_space.sample()), drawn on the device
    # outside the timed event pairs
    g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
    act_buf = torch.empty((n, 2), dtype=torch.float32, device=dev)
    obs, rew, cost, done = env._obs, env._reward, env._cost, env._done
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def step_dev(hh):
        act_buf.uniform_(-1.0, 1.0, generator=g)
        L.check(L.L.sag_step(hh, p(act_buf), p(obs), p(rew), None, p(cost), p(done), sp))

    def ev():
        return torch.cuda.Event(enable_timing=True)

    # ---- warm-up: W steps of a throw-away episode, then a reset so that the timed episode starts at phase 0
    for _ in range(W):
        step_dev(h)
    L.check(L.L.sag_reset(h, None, 0, 0, sp))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()

    # ---- value: stratified timed steps over whole episodes, untimed fast-forward in between
    timed, ff_blocks, reset_evs = [], [], []
    t_wall0 = time.perf_counter()
    l0 = launches_now(h)
    timed_launches = 0
    last_out = None
    for ep_win in ep_windows:
        t = 0
        for (a, ln) in ep_win + [(EPISODE, 0)]:
            if a > t:  # fast-forward (warm L2, timed as one block for the value_l2_warm extra)
                e0, e1 = ev(), ev()
                e0.record(stream)
                for _ in range(a - t):
                    step_dev(h)
                e1.record(stream)
                ff_blocks.append((t, a - t, e0, e1))
            for k in range(ln):
                act_buf.uniform_(-1.0, 1.0, generator=g)
                flush.zero_()  # L2 flush, outside the event pair
                e0, e1 = ev(), ev()
                lc = launches_now(h)
                e0.record(stream)
                L.check(L.L.sag_step(h, p(act_buf), p(obs), p(rew), None, p(cost), p(done), sp))
                e1.record(stream)
                timed_launches += launches_now(h) - lc
                timed.append((a + k, e0, e1))
                if args.dump_outputs and len(timed) == K:  # the last timed step: keep its outputs before the reset
                    last_out = [x.clone() for x in (obs, rew, cost, done)]
            t = a + ln
        e0, e1 = ev(), ev()
        flush.zero_()
        e0.record(stream)
        L.check(L.L.sag_reset(h, None, 0, 0, sp))  # episode end: layout rejection sampling for all envs
        e1.record(stream)
        reset_evs.append((e0, e1))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_wall1 = time.perf_counter()
    # the clocks of the timed region are in; stop polling nvidia-smi before the end-to-end leg (its queries take driver
    # locks that now and then stall a synchronous host call for milliseconds)
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    launches_total = launches_now(h) - l0
    ms = [(ph, a.elapsed_time(b)) for ph, a, b in timed]
    reset_ms = sum(a.elapsed_time(b) for a, b in reset_evs) / len(reset_evs)
    steps_ms = float(sum(m for _, m in ms))
    total_ms = steps_ms + K * reset_ms / EPISODE
    ff_steps = sum(c for _, c, _, _ in ff_blocks)
    ff_ms = float(sum(a.elapsed_time(b) for _, _, a, b in ff_blocks))
    t = torch.tensor([total_ms, steps_ms, reset_ms, ff_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, steps_ms, reset_ms, ff_ms = (float(x) for x in t)
    value = world * n * K / (total_ms * 1e-3)
    value_warm = world * n * ff_steps / (ff_ms * 1e-3) if ff_steps else None
    win_ms = []
    i = 0
    for ep_win in ep_windows:
        for (a, ln) in ep_win:
            if ln:
                w = [m for _, m in ms[i:i + ln]]
                win_ms.append({"phase": a, "steps": ln, "ms_per_step": float(sum(w) / ln)})
            i += ln
    if last_out is not None and rank == 0:
        dump_outputs(args.dump_outputs, *last_out)
        del last_out

    # ---- optional extra: episodes staggered over all 1000 phases (every step some envs auto-reset)
    stagger = None
    if args.stagger:
        env_s = BatchedSafeAdaptationGym("xmls/%s.xml" % cfg["robot"], num_envs=n, device=dev, env_id_base=rank * n,
                                         max_episode_steps=EPISODE)
        env_s.seed(666)
        env_s.set_task([task_objs[(rank * n + e) % len(task_objs)] for e in range(n)])
        hs = env_s._h
        # spread the step counters: env e has already done (e mod 1000) steps of its episode after a 1000-step run-in
        for _ in range(EPISODE):
            step_dev(hs)
        ti = env_s.get_field("task_i32")
        ti[6, :n] = (torch.arange(n, device=dev) % EPISODE).to(torch.int32)
        env_s.set_field("task_i32", ti)
        for _ in range(EPISODE):  # run-in: one full period with auto-reset so that phases are mixed
            step_dev(hs); L.check(L.L.sag_reset(hs, None, 1, 0, sp))
        torch.cuda.synchronize()
        Ks = min(K, 200)
        e0, e1 = ev(), ev()
        e0.record(stream)
        for _ in range(Ks):
            step_dev(hs); L.check(L.L.sag_reset(hs, None, 1, 0, sp))
        e1.record(stream)
        torch.cuda.synchronize()
        stagger = {"value": world * n * Ks / (e0.elapsed_time(e1) * 1e-3), "steps": Ks,
                   "note": "warm L2, step + auto-reset of the ~n/1000 envs that expire every step"}
        env_s.close()

    # ---- end to end through the C ABI with pinned host buffers, on a second handle: one episode, the first episode's strata
    e2e = None
    if not args.no_e2e:
        env2 = make_env()
        h2 = env2._h
        od = env.obs_dim
        act_h = torch.empty((n, 2), dtype=torch.float32).pin_memory()

        class _Raw:  # the four output buffers: one pinned block from the library, laid out for a single D2H copy per step
            def __init__(self, ptr):
                self.ptr = ptr

            def data_ptr(self):
                return self.ptr
        ptrs = [C.c_void_p() for _ in range(4)]
        L.check(L.L.sag_host_alloc_outputs(h2, *[C.byref(x) for x in ptrs]))
        obs_h, rew_h, cost_h, done_h = (_Raw(x.value) for x in ptrs)
        cpu_gen = torch.Generator(); cpu_gen.manual_seed(99 + rank)
        act_h.uniform_(-1, 1, generator=cpu_gen)
        torch.cuda.synchronize()
        for _ in range(W):
            L.check(L.L.sag_step_host(h2, p(act_h), p(obs_h), p(rew_h), p(cost_h), p(done_h)))
        L.check(L.L.sag_reset_host(h2, None, 0, 0, None))
        if world > 1:
            dist.barrier()
        te, ke = 0.0, 0
        t = 0
        for (a, ln) in windows:
            for _ in range(a - t):
                step_dev(h2)
            torch.cuda.synchronize()
            for _ in range(ln):
                act_h.uniform_(-1, 1, generator=cpu_gen)   # the host policy's work is not timed
                t0 = time.perf_counter()
                L.check(L.L.sag_step_host(h2, p(act_h), p(obs_h), p(rew_h), p(cost_h), p(done_h)))  # H2D + kernels + D2H + sync
                te += time.perf_counter() - t0
                ke += 1
            t = a + ln
        for _ in range(EPISODE - t):
            step_dev(h2)
        torch.cuda.synchronize()
        # episode end: env.reset() through the host API (layouts + first observation to the host).  The first call -- the one
        # that follows the episode -- is what is charged; two more are recorded next to it (a large gap between them would be
        # a stall such as the local-memory re-size the library now avoids, sag_kernels.cu Ops::setup)
        resets = []
        for _ in range(3):
            t0 = time.perf_counter()
            L.check(L.L.sag_reset_host(h2, None, 0, 0, p(obs_h)))
            resets.append(time.perf_counter() - t0)
        t_reset_e2e = resets[0]
        te_total = te + ke * t_reset_e2e / EPISODE
        t = torch.tensor([te_total], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        te_total = float(t[0])
        d2h = n * (od * 4 + 8 + 1 + 1)
        # host ceiling: all ranks pull one step's outputs to pinned memory at the same time, back to back (tools/probe_d2h.py)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        secs = C.c_double()
        L.check(L.L.sag_probe_d2h(h2, d2h, 40, C.byref(secs)))
        # sum over ranks of each rank's own copy rate while all ranks copy (ranks behind different PCIe switches get
        # different shares, so total bytes / slowest rank's time would understate the aggregate)
        tc = torch.tensor([d2h * 40 / secs.value / 1e9], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tc, op=dist.ReduceOp.SUM)
        ceiling_gbs = float(tc[0])
        e2e_value = world * n * ke / te_total
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * 2 * 4,
               "d2h_bytes_per_step": d2h, "steps": ke, "reset_ms": 1e3 * t_reset_e2e, "reset_ms_samples": [1e3 * r for r in resets],
               "d2h_gbs": e2e_value / n * d2h / 1e9, "host_ceiling_gbs": ceiling_gbs,
               "host_ceiling_frac": (e2e_value / n * d2h / 1e9) / ceiling_gbs,
               "host_ceiling_note": ("ceiling = sum of the ranks' copy rates while ALL ranks copy one step's outputs device -> pinned host back to "
                                     "back; with several ranks the e2e steps are not in lockstep, so their copies contend less than the probe's"),
               "binding": binding,
               "api": "sag_step_host (C ABI; one pinned output block, a single D2H copy per step); one episode, timed in the windows "
                      "of `value`'s first episode"}
        L.L.sag_host_free(C.c_void_p(ptrs[0].value))
        env2.close()

    # ---- per-task statistics: the only collective on this path (NCCL all-reduce of a [14,3] fp64 buffer)
    stats = env.task_stats(reset=True)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    stats = stats.cpu().numpy()

    if rank == 0:
        peak, peak_src = peaks()
        avg_s = total_ms * 1e-3 / K
        achieved = cfg["b_alg"] * n / avg_s / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp) and args.config == "point_gtg":
            try:
                traffic = json.load(open(tp)).get("step_dram_bytes_per_launch")
            except Exception:
                traffic = None
        first_s = win_ms[0]["ms_per_step"] * 1e-3
        line = {
            "metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["workload"], "envs_per_gpu": n, "global_envs": world * n, "parallelism": f"env-shard x{world}",
                       "l2": "flushed before every timed step (256 MiB memset outside the event pair)", "action_noise": 0.01,
                       "episode_phase": (f"stratified over {n_ep} whole {EPISODE}-step episode(s), {K} timed steps: per episode "
                                         f"{len(windows)} windows of {min(ln for w in ep_windows for _, ln in w)}.."
                                         f"{max(ln for w in ep_windows for _, ln in w)} steps at phases "
                                         f"{[[a for a, _ in w] for w in ep_windows]} (one list per episode), untimed fast-forward "
                                         f"in between, + reset {reset_ms:.3f} ms amortised / {EPISODE}")},
            "ms_per_step_windows": win_ms, "reset_ms": reset_ms,
            "value_l2_warm": value_warm,
            "value_l2_warm_note": "the fast-forward steps between the windows (no flush, back to back), whole-episode coverage",
            "e2e": e2e,
            "gpu_launches": timed_launches + n_ep, "gpu_launches_incl_fast_forward": launches_total,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "kernel": "fused step (free-motion kernel + contact kernel), whole-episode average",
                         "b_alg_per_env_step": cfg["b_alg"], "peak_source": peak_src,
                         "frac_quiet_phase": cfg["b_alg"] * n / first_s / 1e9 / peak},
            "clocks": clocks,
            "episode_stats": {t: {"sum_return": float(stats[TASKS[t].task_id, 0]), "sum_cost": float(stats[TASKS[t].task_id, 1]),
                                  "episodes": float(stats[TASKS[t].task_id, 2])} for t in cfg["tasks"]},
            "wall_s_timed_region": t_wall1 - t_wall0,
        }
        if stagger:
            line["staggered_episodes"] = stagger
        if not args.no_cpu_baseline and world == 1:
            cores = os.cpu_count() or 1
            ne = (16 if cfg["robot"] == "point" else 2) * cores
            r, c, dt = cpu_oracle_rate(cfg, ne, EPISODE, cores)
            line["cpu_baseline"] = {"value": r, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{ne} envs x {EPISODE} steps (whole episodes) = {c} env-steps in {dt:.1f}s, oracle port "
                                              "(C, pthreads); the reference's MuJoCo stack is not installable here"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
