"""
Cost of the wide action heads at C4-shaped networks (actor 376-256^3-P, critic 376-256^3-1, Tanh, B = 512), launch
chain:
  - device time per minibatch step for Discrete(64 | 65 | 362 | 4672) and Box(64 | 65 | 256), alternating runs;
  - per-launch device time of one step from torch.profiler (kernel names as compiled), so the loss kernel stands beside
    the head layer's forward and backward grouped-GEMM launches;
  - get_rollout_actions per call at E = 64 for Discrete(4672): wall time, and the host Exp(1) draws alone;
  - the card's name and power limit, read in the same run.

    python scratch/wide_head_cost.py [--epochs 10] [--repeats 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

OBS, HIDDEN, B, T, E = 376, 256, 512, 64, 128


def build(kind, width, envs):
    from helpers import ACT_MODULES, run_device_rollout
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    from ppo_and_friends_b200.spaces import Box, Discrete
    from ppo_and_friends_b200.synthetic import make_rollout
    ro = make_rollout(seed=5, T=T, E=envs, obs_dim=OBS, act_dim=width, n_discrete=width if kind == "Discrete" else 0,
                      max_ts_per_ep=32, obs_scale=False)
    space = Discrete(width) if kind == "Discrete" else Box(-1.0, 1.0, (width,))
    torch.manual_seed(0)
    pol = PPOPolicy("pol", space, Box(-np.inf, np.inf, (OBS,)), Box(-np.inf, np.inf, (OBS,)), envs_per_proc=envs,
                    actor_kw_args=dict(activation=ACT_MODULES["tanh"](), hidden_size=HIDDEN, hidden_depth=3),
                    critic_kw_args=dict(activation=ACT_MODULES["tanh"](), hidden_size=HIDDEN, hidden_depth=3))
    pol.register_agent("agent0")
    pol.finalize({"global status": {"iteration": 0, "timesteps": 0}}, torch.device("cuda"))
    return pol, ro, run_device_rollout(pol, ro)


def step_time(kind, width, epochs, repeats):
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    pol, ro, ds = build(kind, width, E)
    state = PPOUpdateState({"pol": pol}, batch_size=B, epochs_per_iter=1)
    loader = _Loader(ds, B)
    for _ in range(3):                                                     # warm-up: graph capture, module loads
        ppo_batch_train(state, loader, "pol")
    steps = len(ds) // B
    times = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(epochs):
            ppo_batch_train(state, loader, "pol")
        t1.record()
        torch.cuda.synchronize()
        times.append(t0.elapsed_time(t1) * 1e3 / (epochs * steps))
    return dict(space=f"{kind}({width})", steps_per_epoch=steps, us_per_step=[round(t, 1) for t in times])


def launch_profile(kind, width):
    """Mean device time of every launch position of a full minibatch step (graphs off: one kernel per launch)."""
    from torch.profiler import ProfilerActivity, profile
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    os.environ["PPOAF_NO_GRAPH"] = "1"
    try:
        pol, ro, ds = build(kind, width, E)
        state = PPOUpdateState({"pol": pol}, batch_size=B, epochs_per_iter=1)
        loader = _Loader(ds, B)
        ppo_batch_train(state, loader, "pol")
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                ppo_batch_train(state, loader, "pol")
            torch.cuda.synchronize()
    finally:
        os.environ.pop("PPOAF_NO_GRAPH", None)
    ks = sorted([e for e in prof.events() if e.device_type.name == "CUDA"], key=lambda e: e.time_range.start)
    # a step runs from the first grouped-GEMM launch after an Adam launch to the next Adam launch
    steps, cur = [], []
    for e in ks:
        cur.append(e)
        if "adam" in e.name.lower():
            if any("loss" in k.name for k in cur):
                steps.append([k for k in cur if "gemm" in k.name or "loss" in k.name or "adam" in k.name])
            cur = []
    n = min(len(s) for s in steps)
    steps = [s for s in steps if len(s) == n]
    rows = []
    for p in range(n):
        name = steps[0][p].name
        rows.append(dict(pos=p, kernel=name.split("(")[0][-40:], us=round(float(np.mean(
            [s[p].time_range.elapsed_us() for s in steps])), 1)))
    return dict(space=f"{kind}({width})", steps_profiled=len(steps), launches=rows)


def rollout_time(width, calls=200):
    pol, ro, _ = build("Discrete", width, 64)
    obs = ro.obs["agent0"][0]
    for _ in range(10):
        pol.get_rollout_actions(obs)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        pol.get_rollout_actions(obs)
    wall = (time.perf_counter() - t0) / calls
    t0 = time.perf_counter()
    for _ in range(calls):
        torch.empty(64, width, dtype=torch.float32).exponential_(1)
    draws = (time.perf_counter() - t0) / calls
    return dict(space=f"Discrete({width})", E=64, us_per_call=round(wall * 1e6, 1), host_draws_us=round(draws * 1e6, 1),
                rest_us=round((wall - draws) * 1e6, 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps(dict(gpu=smi[0] if smi else "unknown")), flush=True)
    spaces = [("Discrete", 64), ("Discrete", 65), ("Discrete", 362), ("Discrete", 4672), ("Box", 64), ("Box", 65),
              ("Box", 256)]
    for _ in range(2):                                                     # two alternating passes: run-to-run spread
        for kind, width in spaces:
            print(json.dumps(step_time(kind, width, args.epochs, args.repeats)), flush=True)
    for kind, width in (("Discrete", 64), ("Discrete", 65), ("Discrete", 4672), ("Box", 256)):
        print(json.dumps(launch_profile(kind, width)), flush=True)
    print(json.dumps(rollout_time(4672)), flush=True)


if __name__ == "__main__":
    main()
