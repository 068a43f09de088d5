"""
Device time per minibatch step of the Bernoulli head next to the Categorical head, at C5-shaped networks
(actor 18-128^3-15, critic 54-256^3-1, Tanh, B = 128): MultiBinary(15) vs Discrete(15), on both step engines
(the launch chain and the persistent fused kernel).  Prints one JSON line per (engine, head) and the card it ran on.

    python scratch/multi_binary_cost.py [--epochs 20] [--repeats 3]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def build_policy(head, ro):
    from helpers import ACT_MODULES
    from ppo_and_friends_b200.policies.ppo_policy import PPOPolicy
    from ppo_and_friends_b200.spaces import Box, Discrete, MultiBinary
    space = MultiBinary(15) if head == "binary" else Discrete(15)
    pol = PPOPolicy("pol", space, Box(-np.inf, np.inf, (18,)), Box(-np.inf, np.inf, (54,)), envs_per_proc=ro.E,
                    actor_kw_args=dict(activation=ACT_MODULES["tanh"](), hidden_size=128, hidden_depth=3),
                    critic_kw_args=dict(activation=ACT_MODULES["tanh"](), hidden_size=256, hidden_depth=3))
    pol.register_agent("agent0")
    pol.finalize({"global status": {"iteration": 0, "timesteps": 0}}, torch.device("cuda"))
    return pol


def measure(engine, head, epochs, repeats):
    from helpers import run_device_rollout
    from ppo_and_friends_b200.ppo import PPOUpdateState, _Loader, ppo_batch_train
    from ppo_and_friends_b200.synthetic import make_rollout
    os.environ["PPOAF_STEP"] = engine
    ro = make_rollout(seed=5, T=64, E=128, obs_dim=18, critic_obs_dim=54, act_dim=15, max_ts_per_ep=32, obs_scale=False)
    rng = np.random.default_rng(6)
    if head == "binary":
        acts = rng.integers(0, 2, size=(ro.T, ro.E, 15)).astype(np.float32)
    else:
        acts = rng.integers(0, 15, size=(ro.T, ro.E, 1)).astype(np.int64)
    ro.raw_actions["agent0"] = acts
    ro.actions["agent0"] = acts.copy()
    torch.manual_seed(0)
    pol = build_policy(head, ro)
    ds = run_device_rollout(pol, ro)
    state = PPOUpdateState({"pol": pol}, batch_size=128, epochs_per_iter=1)
    loader = _Loader(ds, 128)
    for _ in range(3):                                                     # warm-up: graph capture, module loads
        ppo_batch_train(state, loader, "pol")
    steps = len(ds) // 128
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
    return dict(engine=engine, head=head, fused_engine=bool(pol._engine.fused), steps_per_epoch=steps,
                us_per_step=[round(t, 2) for t in times])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps(dict(gpu=smi[0] if smi else "unknown")))
    for engine in ("chain", "fused"):
        for head in ("discrete", "binary", "discrete", "binary"):           # alternating: run-to-run spread
            print(json.dumps(measure(engine, head, args.epochs, args.repeats)), flush=True)


if __name__ == "__main__":
    main()
